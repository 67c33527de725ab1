// Host engine of libsnn_b200.so — a from-scratch C++ counterpart of ShaderNN's model loading / graph building /
// execution stack, keeping its names so the mapping to the reference is one-to-one:
//
//   snn::dp::ModelParser            core/src/ic2/modelparser.{h,cpp}      JSON (+ sidecar .bin) model reader
//   snn::dp::<Op>Desc / <Op>Layer   core/src/ic2/<op>.{h,cpp}             per-op descs, dims, padding rules
//   snn::dp::registerLayer / createLayerInstance   layerFactory.{h,cpp}   string -> creator registry + aliases
//   snn::dp::loadFromJsonModel / generateInferenceGraph   dp.{h,cpp}      DAG wiring, Kahn toposort, dims
//   snn::MixedInferenceCore         core/inc/snn/core.h, core/src/ic2/core.cpp   stage list, init, run
//   snn::dp::CudaBackend            (new) backend.h's DeviceBackend role  streams, graphs, timers, dumps
//
// What differs by design: a batch dimension N, NHWC split-fp16 device tensors, weights BN-folded and packed once
// into a single device arena, one CUDA kernel launch per layer (fewer with fusion), optional CUDA-graph replay.
#pragma once

#include <algorithm>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../snnb_internal.h"
#include "json.h"

namespace snn {

struct SNNModelOutputBoxes { // yololayer.cpp:219-225 rows {class, score, x, y, w, h}
    std::vector<std::vector<float>> rows;
};

namespace dp {

// -------------------------------------------------------------------------------------------------------------
// ModelParser (modelparser.h:30-157). Reads "numLayers", "Layer_<i>", optional "inputRange"; when
// numLayers.bin_file_name is present the weights stream from that sidecar file (raw LE fp32, layer order) which is
// looked up next to the JSON file.
// -------------------------------------------------------------------------------------------------------------
class ModelParser {
public:
    explicit ModelParser(const std::string& fileName);
    ~ModelParser();
    int getLayerCount() const;
    std::string getLayerName(int layerId) const; // "type", or "name" when type == "Lambda" (modelparser.cpp:78-86)
    int getNumInbound(int layerId) const;
    std::vector<int> getInboundLayerId(int layerId) const;
    int getInputPlanes(int layerId) const;
    int getOutputPlanes(int layerId) const;
    bool isInputRange01() const;
    const json::Value& layer(int layerId) const;
    bool isBinWeight() const { return binFile != nullptr; }
    // next `count` floats of the sidecar stream
    void readBin(float* dst, size_t count);
    const std::string& fileName() const { return _fileName; }

private:
    std::string _fileName;
    json::ValuePtr _root;
    FILE* binFile = nullptr;
};

// Padding spec as the parser leaves it: four strings, either all digits or a keyword ("same"/"valid"/"none")
// (modelparser.cpp:584-609), plus the conv "mode".
int padModeId(const std::string& mode); // SNNB_PAD_* of a padding mode string (conv2dVulkan.cpp:73-80)
struct PaddingSpec {
    std::string t = "valid", b = "valid", l = "valid", r = "valid";
    std::string mode; // "constant" | "replicate" | "reflect" | "" (unset)
    void parse(const json::Value& layerObj, bool readMode);
    // conv2d.cpp:39-74 / separableconvolution.cpp:27-62 / maxpool2d.cpp:37-72: {T, B, L, R}
    void offsets(int kernelSize, bool evenKernelTopLeftMinusOne, uint32_t (&offs)[4]) const;
    bool validLike() const { return t == "0" || t == "valid" || t == "none"; }
};

struct Dims {
    uint32_t width = 0, height = 0, depth = 0; // depth = channels here (the reference's IODesc carries both ceil(C/4) and C)
};

struct ActivationSpec {
    int id      = SNNB_ACT_NONE;
    float alpha = 0.0f;
    // Accepts every spelling the reference uses (SURVEY Q12): conv "leakyRelu", add/activation/dense "leaky_relu",
    // CPU map "SiLU"/"softmax"/"identity"/""; anything unknown is identity (conv2dVulkan.cpp:58-72).
    static int fromString(const std::string& s);
};

struct ExecOptions; // below

// -------------------------------------------------------------------------------------------------------------
// GenericModelLayer (genericlayer.h:60-139): graph node + execution unit.
// -------------------------------------------------------------------------------------------------------------
class GenericModelLayer {
public:
    virtual ~GenericModelLayer() {}
    std::string name;      // "<file> layer [NN] <Type>" (dp.cpp:135)
    std::string typeName;  // registry name after aliasing
    int layerId = -1;
    std::vector<GenericModelLayer*> prevLayers, nextLayers;
    std::vector<Dims> inputDims;
    uint32_t numInputPlanes = 0, numOutputPlanes = 0;
    bool isInputLayer = false;

    // genericlayer.cpp:64-90 default: out = uint32(scale*in + translate) per axis, depth = max input depth
    virtual void getOutputDims(uint32_t& width, uint32_t& height, uint32_t& depth) const;
    struct Transform { float scaleW = 1, scaleH = 1, transW = 0, transH = 0; };
    virtual Transform getOutputScaleDimAdjustment() const { return Transform(); }

    // ---- execution ----
    // fold/pack this layer's weights on the host (no device work); empty for weightless layers
    virtual void packWeights(snnb::PackedHost&) {}
    snnb_weights weights; // points into the model's arena after init
    std::vector<snnb_tensor*> inputs;
    snnb_tensor* output = nullptr;
    // GenericModelLayer::run -> RenderPass::run (genericlayer.cpp:39-62): enqueue this layer's kernel(s)
    virtual int run(snnb_context* ctx, const ExecOptions& opt) = 0;
    // fusion bookkeeping (engine-level; see MixedInferenceCore::init)
    bool fusedAway          = false;      // produces nothing itself (its work happens inside another layer)
    snnb_tensor* residual   = nullptr;    // Conv2D: tensor added before the activation (fused Add)
    int fusedAct            = -1;         // Conv2D: activation taken over from a fused Add (-1 = own)
    float fusedAlpha        = 0.0f;
    float* scratch          = nullptr;    // per-layer device scratch (InstanceNorm stats)
    size_t scratchBytes() const { return _scratchBytes; }

protected:
    size_t _scratchBytes = 0;
};

// A layer supplied through the C-ABI (snnb_register_layer): dims and launches are the host's callbacks.
class PluginLayer : public GenericModelLayer {
public:
    snnb_layer_impl impl {};
    ~PluginLayer() override {
        if (impl.destroy) impl.destroy(impl.user);
    }
    void getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const override;
    int run(snnb_context* ctx, const ExecOptions& opt) override;
};

typedef GenericModelLayer* (*LayerCreator)(ModelParser&, int);
void initLayerRegisty();
void registerLayer(const std::string& layerName, LayerCreator creator);
GenericModelLayer* createLayerInstance(std::string layerName, ModelParser& parser, int i);

// -------------------------------------------------------------------------------------------------------------
// Layers
// -------------------------------------------------------------------------------------------------------------
struct InputLayerDesc {
    uint32_t inputWidth = 0, inputHeight = 0, inputChannels = 0, inputIndex = 0;
    void parse(ModelParser& parser, int layerId); // modelparser.cpp:480-497
};
class InputLayerLayer : public GenericModelLayer {
public:
    InputLayerDesc _desc;
    void getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const override;
    int run(snnb_context*, const ExecOptions&) override { return 0; }
};

struct GenericConvDesc {
    uint32_t kernelSize = 1, stride = 1;
    PaddingSpec padding;
    ActivationSpec activation;
    std::string activationName;
    std::vector<float> weights; // Conv2D: OIHW; depthwise: [C][k][k]
    std::vector<float> biases;  // empty when useBias is not "True"
    bool useBatchNormalization = false;
    std::map<std::string, std::vector<float>> batchNormalization; // gamma beta movingMean movingVariance
};
struct Conv2DDesc : GenericConvDesc {
    void parse(ModelParser& parser, int layerId); // modelparser.cpp:574-781
};
class Conv2DLayer : public GenericModelLayer {
public:
    Conv2DDesc _desc;
    int algo = SNNB_ALGO_AUTO;
    // Replicate / reflect padding on the tensor path: the TMA unit can only zero-fill, so the engine materialises the
    // padded input once (pad kernel, vk_pad.comp semantics) and runs the tcgen05 kernel over it with zero padding.
    snnb_tensor* prepadded = nullptr;
    // Stride-2 stem with <= 4 input channels reading a model input: the input tensor carries a compact 4-channel copy
    // (snnb_tensor::feed_hi) and the weights get the matching K order (FeedPlan, kernels_umma.cu conv_rowwin_kernel feed mode).
    bool feedInput = false;
    // Projection shortcut folded into this convolution's K loop (fusion pass in MixedInferenceCore::init): `shortcut` is the 1x1 conv
    // whose product this layer adds, reading `shortcutIn`; the shortcut layer itself launches nothing and points back via `foldedInto`.
    Conv2DLayer* shortcut    = nullptr;
    Conv2DLayer* foldedInto  = nullptr;
    snnb_tensor* shortcutIn  = nullptr;
    bool wantsPrepad(const snnb_tensor* in, const snnb_tensor* out, int convAlgo, int& ph, int& pw) const;
    Transform getOutputScaleDimAdjustment() const override; // conv2d.cpp:102-113
    void getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const override;
    void packWeights(snnb::PackedHost& p) override;
    int run(snnb_context* ctx, const ExecOptions& opt) override;
};
struct SeparableConv2DDesc : GenericConvDesc {
    void parse(ModelParser& parser, int layerId); // modelparser.cpp:783-985
};
class SeparableConv2DLayer : public GenericModelLayer { // depthwise (the name is historical)
public:
    SeparableConv2DDesc _desc;
    void getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const override; // separableconvolution.cpp:77-86
    void packWeights(snnb::PackedHost& p) override;
    int run(snnb_context* ctx, const ExecOptions& opt) override;
};
struct PoolDesc {
    uint32_t kernelSize = 1, stride = 1;
    PaddingSpec padding;
    void parseMax(ModelParser& parser, int layerId); // modelparser.cpp:304-371
    void parseAvg(ModelParser& parser, int layerId); // modelparser.cpp:373-397
};
class PoolingLayer : public GenericModelLayer { // MaxPooling2D / AveragePooling2D
public:
    PoolDesc _desc;
    bool isAvg = false;
    Transform getOutputScaleDimAdjustment() const override; // maxpool2d.cpp:26-35, avgpool2d.cpp:21-30
    int run(snnb_context* ctx, const ExecOptions& opt) override;
};
class AdaptiveAvgPool2dLayer : public GenericModelLayer { // adaptiveavgpool2d.h (GL-only in the reference): pool -> pool x pool
public:
    uint32_t poolSize = 1;
    void getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const override;
    int run(snnb_context* ctx, const ExecOptions& opt) override;
};
class AddLayer : public GenericModelLayer { // addlayer.h:27-46
public:
    ActivationSpec activation;
    int run(snnb_context* ctx, const ExecOptions& opt) override;
};
class BatchNormalizationLayer : public GenericModelLayer { // batchnorm.h:28-50
public:
    std::map<std::string, std::vector<float>> batchNormalization;
    ActivationSpec activation;
    void packWeights(snnb::PackedHost& p) override;
    int run(snnb_context* ctx, const ExecOptions& opt) override;
};
class InstanceNormLayer : public GenericModelLayer { // instancenorm.h:28-54
public:
    std::vector<float> gamma, beta;
    ActivationSpec activation;
    void packWeights(snnb::PackedHost& p) override;
    int run(snnb_context* ctx, const ExecOptions& opt) override;
    void setScratch() { _scratchBytes = 0; }
    void computeScratch(int n) { _scratchBytes = snnb::instnorm_scratch_floats(n, snnb::round_up((int) numOutputPlanes, 8)) * sizeof(float); }
};
class ActivationLayer : public GenericModelLayer { // activation.h:27-48 (creatable, not registered in the reference)
public:
    ActivationSpec activation;
    int run(snnb_context* ctx, const ExecOptions& opt) override;
};
class DenseLayer : public GenericModelLayer { // denselayer.cpp:27-54
public:
    std::vector<float> kernel; // flat, [out][in]
    std::vector<float> biases;
    ActivationSpec activation;
    uint32_t units = 0;
    void getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const override;
    void packWeights(snnb::PackedHost& p) override;
    int run(snnb_context* ctx, const ExecOptions& opt) override;
    snnb_tensor* flat = nullptr; // staging when the input is not 1x1
    GenericModelLayer* gapSource = nullptr; // fused head: global average pool of this layer's output feeds the Dense (core.cpp, fusion 4)
};
class FlattenLayer : public GenericModelLayer { // flattenlayer.cpp:29-62 (CPU flavour: HWC order)
public:
    ActivationSpec activation;
    void getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const override;
    int run(snnb_context* ctx, const ExecOptions& opt) override;
};
class ConcatenateLayer : public GenericModelLayer { // concatenation.h:25-40
public:
    void getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const override;
    int run(snnb_context* ctx, const ExecOptions& opt) override;
};
class UpSampling2DLayer : public GenericModelLayer { // upsampling2d.h:26-47
public:
    float scale = 1.0f;
    std::string interpolationType = "nearest";
    Transform getOutputScaleDimAdjustment() const override { return Transform {scale, scale, 0.0f, 0.0f}; }
    int run(snnb_context* ctx, const ExecOptions& opt) override;
};
class PadLayer : public GenericModelLayer { // padlayer.{h,cpp}
public:
    PaddingSpec padding;
    std::string mode = "constant"; // the reference parser never overwrites it (modelparser.cpp:1112-1113 drops the argument)
    Transform getOutputScaleDimAdjustment() const override; // padlayer.cpp:60-68
    int run(snnb_context* ctx, const ExecOptions& opt) override;
};
class SubpixelLayer : public GenericModelLayer { // subpixelmerge.h:26-47
public:
    uint32_t kernelSize = 2;
    void getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const override;
    int run(snnb_context* ctx, const ExecOptions& opt) override;
};
class YOLOLayer : public GenericModelLayer { // yololayer.{h,cpp}: host decode + NMS of two heads
public:
    void getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const override;
    int run(snnb_context*, const ExecOptions&) override { return 0; } // executed by the core after the device pass (candidates + host NMS)
    // all-host decode (downloads both heads): the fallback when an image has more candidates than the device list holds
    int decode(snnb_context* ctx, std::vector<SNNModelOutputBoxes>& perImage);
    // device threshold + compaction into `devCounts` / `devCand` ([N] ints, [N][YOLO_MAX_CAND][8] floats), asynchronous
    // one slot per (image, cell, anchor) of both heads: the list can never overflow, whatever the scores. Layout: 32-byte header
    // (word 0 = number of candidates) + rows of 8 floats. The host copies the header and the first YOLO_HEAD_ROWS rows with every
    // submission; the (rare) rest is fetched in wait().
    static constexpr int YOLO_HEAD_ROWS = 2048;
    int maxCand() const { return inputs.size() < 2 ? 0 : inputs[0]->n * (inputs[0]->h * inputs[0]->w + inputs[1]->h * inputs[1]->w) * 3; }
    size_t candidateBytes() const { return 32 + (size_t) maxCand() * 8 * sizeof(float); }
    size_t headBytes() const { return 32 + (size_t) std::min(maxCand(), YOLO_HEAD_ROWS) * 8 * sizeof(float); }
    int enqueueCandidates(snnb_context* ctx, void* devBuf);
    // host part on the downloaded buffer: exact score formula, confidence threshold, score sort, NMS (yololayer.cpp:56-164).
    // Returns 0, or -1 when some image overflowed the candidate list (caller falls back to decode()).
    int finishDecode(const void* hostBuf, const void* devBuf, std::vector<SNNModelOutputBoxes>& perImage) const;
};

// -------------------------------------------------------------------------------------------------------------
// dp.h: model loading + graph generation
// -------------------------------------------------------------------------------------------------------------
struct ShaderGenOptions { // layeroption.h:27-48, trimmed to what a CUDA backend can honour, + batch
    uint32_t desiredInputWidth = 0, desiredInputHeight = 0; // desiredInput[0] (dp.cpp:505-507)
    uint32_t batch             = 1;
    int convAlgo               = SNNB_ALGO_AUTO;
    bool fuse                  = false;
    bool useCudaGraph          = false;
    int precision              = SNNB_PRECISION_FP32X3; // layeroption.h:43 preferrHalfPrecision <-> SNNB_PRECISION_FP16
};
struct ExecOptions {
    int convAlgo  = SNNB_ALGO_AUTO;
    int precision = SNNB_PRECISION_FP32X3;
};

std::vector<std::shared_ptr<GenericModelLayer>> loadFromJsonModel(const std::string& fileName); // dp.cpp:115-167
// Kahn topological sort over nextLayers (dp.cpp:389-429), dims propagation (dp.cpp:432-640).
struct InferenceGraph {
    std::vector<GenericModelLayer*> sorted; // execution order, inputs first
    std::vector<Dims> outputDims;           // per sorted layer
};
InferenceGraph generateInferenceGraph(const std::vector<std::shared_ptr<GenericModelLayer>>& layers, const ShaderGenOptions& options);

} // namespace dp

// -------------------------------------------------------------------------------------------------------------
// MixedInferenceCore (core.h:66-146, core.cpp): owns the stages' tensors, the weight arena, the CUDA graph.
// -------------------------------------------------------------------------------------------------------------
class MixedInferenceCore {
public:
    ~MixedInferenceCore();
    static std::unique_ptr<MixedInferenceCore> create(snnb_context* ctx, const std::string& modelFileName, const dp::ShaderGenOptions& options,
                                                      std::string& err);
    // forward pass only (inputs already resident in the InputLayers' tensors); asynchronous
    int forward();
    // host -> input tensor idx (async H2D + split kernel)
    int setInput(int idx, const float* hostNHWC);
    // output idx -> host NHWC (merge kernel + D2H, synchronous)
    int getOutput(int idx, float* host, size_t capacityFloats);
    // run(RunParameters) end to end (core.cpp:97-245): H2D, forward, D2H, class index
    int run(const float* hostInput, float* hostOutput, size_t capacityFloats, int* classes1);
    // streaming: double-buffered submit/wait (H2D of batch i+1 overlaps compute of batch i)
    int submit(const float* hostInput, float* hostOutput, size_t capacityFloats, int* classes1, int* ticket);
    // same with a u8 NHWC image batch, normalised on the device as (x - mean[c]) * norm[c] (imageTexture.h:114)
    int submitU8(const uint8_t* hostInput, const float mean[4], const float norm[4], float* hostOutput, size_t capacityFloats, int* classes1, int* ticket);
    int submitImpl(const void* hostInput, bool u8, const float* mean, const float* norm, float* hostOutput, size_t capacityFloats, int* classes1, int* ticket,
                   const snnb_image_io* io = nullptr);
    int submitImage(const snnb_image_io& io, int* ticket);
    int wait(int ticket);
    int layerOutput(int layerId, float* host, size_t capacityFloats);
    int timeLayers(std::vector<float>& ms);
    int dumpOutputs(const std::string& dir);

    snnb_context* ctx = nullptr;
    dp::ShaderGenOptions options;
    std::vector<std::shared_ptr<dp::GenericModelLayer>> layers; // JSON order
    dp::InferenceGraph graph;
    std::vector<dp::GenericModelLayer*> inputLayers, outputLayers;
    std::vector<SNNModelOutputBoxes> boxes; // per image, when the model ends in a YOLO layer
    void* arena       = nullptr;
    size_t arenaBytes = 0;
    int launchesPerForward = 0;
    bool isClassifier = false;
    std::vector<std::string> layerKernels; // per layer (JSON order): the kernel its last timeLayers() pass launched

private:
    bool init(std::string& err);
    int enqueueForward(bool countOnly);
    std::vector<snnb_tensor*> ownedTensors;
    void* scratchArena = nullptr;
    cudaGraph_t cuGraph         = nullptr;
    cudaGraphExec_t cuGraphExec = nullptr;
    float* ioStage   = nullptr; // device fp32 staging for input/output conversion (stable address: graph-safe)
    size_t ioStageBytes = 0;
    int* argmaxDev   = nullptr;
    dp::YOLOLayer* yolo = nullptr;
    void* yoloDev  = nullptr; // device candidate lists of the YOLO decode (counts + [N][YOLO_MAX_CAND][8])
    void* yoloHost = nullptr; // pinned host mirror
    int decodeYolo(void* dev, void* host, bool sync); // candidates kernel + D2H (+ sync + host NMS into `boxes`)
    // streaming state
    static constexpr size_t SMALL_RESULT_BYTES = 64 * 1024;
    struct Slot {
        void* stageResize = nullptr; // device staging of a differently-sized u8 input (grown on demand)
        size_t stageResizeBytes = 0;
        float* stageIn = nullptr;   // device fp32 staging for this slot's input batch
        float* stageOut = nullptr;  // device fp32 staging for output 0
        int* argmax = nullptr;
        cudaEvent_t h2dDone = nullptr, stageFree = nullptr, resultReady = nullptr;
        int* classesHost = nullptr;
        // small classifier results bypass the copy engine: one kernel writes values + arg-max into this mapped pinned block, wait() hands
        // them to the caller's buffers (two ~10 us device->host copy commands less per batch)
        void* smallHost = nullptr;      // cudaHostAlloc'ed, SMALL_RESULT_BYTES
        void* smallDev  = nullptr;      // its device alias
        float* userOut = nullptr;       // where wait() copies the values
        int* userClasses = nullptr;     // ... and the 1-based classes
        size_t userFloats = 0;
        void* yoloDev = nullptr;
        void* yoloHost = nullptr;
        bool busy = false, everUsed = false;
    } slots[2];
    cudaStream_t copyStream = nullptr;
    int nextTicket = 0;
    int ensureStreaming();
};

} // namespace snn
