/*
 * snnb.h — C-ABI of libsnn_b200.so: the B200 (sm_100a) backend for ShaderNN's operator / graph API.
 *
 * This is the drop-in boundary (SURVEY.md §8b): plain C, opaque handles, plain pointers and sizes,
 * `int` status (0 = ok, non-zero = error, message via snnb_last_error()), never throws or aborts
 * across the boundary, no torch types. Everything launches on the context's CUDA stream; calls are
 * asynchronous unless stated. One context per device; no internal threads.
 *
 * Each entry point names the reference interface it replaces (paths relative to the reference repo
 * inferenceengine/shadernn @ 6f3fc8b1). INTEGRATION.md shows the C++ glue a ShaderNN maintainer adds
 * (GpuBackendType::CUDA -> CudaBackend : dp::DeviceBackend, CudaRenderPass : dp::RenderPass).
 *
 * Tensor layout at this boundary: host fp32, either NHWC (N added — the reference is N==1) or the
 * reference's own texture layout "C4HW4" (core/inc/snn/imageTexture.h; element (x,y,c) at
 * (((c/4)*H + y)*W + x)*4 + c%4, demo/common/shaderUnitTest.cpp:87-131). Device storage is private:
 * two fp16 planes (hi, lo = value - hi) in NHWC with the channel pitch padded to 8 — an fp32-faithful
 * (22 significant bits, range +-65504) format that TMA can feed straight to tcgen05 tensor cores (see DESIGN.md).
 */
#ifndef SNNB_H_
#define SNNB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SNNB_VERSION 100

typedef struct snnb_context snnb_context; /* replaces snn::GpuContext + dp::DeviceBackend (core/src/ic2/backend.h:32-91) */
typedef struct snnb_tensor snnb_tensor;   /* replaces snn::ImageTexture device side (core/inc/snn/imageTexture.h:31-352) */
typedef struct snnb_weights snnb_weights; /* replaces InferencePass::_vecWeights/_vecBias/... (core/src/ic2/inferencepass.h:31-59) */
typedef struct snnb_model snnb_model;     /* replaces snn::MixedInferenceCore (core/inc/snn/core.h:66-146) */
typedef struct snnb_timer snnb_timer;     /* replaces snn::DeviceTimer (core/inc/snn/deviceTimer.h) */

/* Activation ids = the Vulkan host's (core/src/ic2/conv2dVulkan.cpp:57-71). SOFTMAX only for Dense. */
enum { SNNB_ACT_NONE = 0, SNNB_ACT_RELU = 1, SNNB_ACT_RELU6 = 2, SNNB_ACT_TANH = 3, SNNB_ACT_SIGMOID = 4, SNNB_ACT_LEAKY_RELU = 5, SNNB_ACT_SILU = 6, SNNB_ACT_SOFTMAX = 7 };
/* Padding modes = conv2dVulkan.cpp:73-80 (0 = unset: out-of-range taps read 0, same as constant). */
enum { SNNB_PAD_NONE = 0, SNNB_PAD_CONSTANT = 1, SNNB_PAD_REPLICATE = 2, SNNB_PAD_REFLECT = 3 };
/* Kernel selection for convolutions. AUTO picks the tcgen05 implicit-GEMM path when the shape allows. TCGEN05_STREAMK also lets the
 * planner cut the K loops of the last partial wave of tiles across all SMs (stream-K; measured slower than whole tiles on ResNet-18's
 * shapes - DESIGN.md 3.4 - so it is not part of AUTO; environment SNNB_SK=1 enables it for every launch). */
enum { SNNB_ALGO_AUTO = 0, SNNB_ALGO_SIMT = 1, SNNB_ALGO_TCGEN05 = 2, SNNB_ALGO_TCGEN05_STREAMK = 3 };
/* Arithmetic / storage precision of the tensor-core convolution path (the reference's counterpart is
 * ShaderGenOptions::preferrHalfPrecision, core/inc/snn/layeroption.h:43: fp32 by default, RGBA16F when set).
 *   FP32X3: activations AND weights as fp16 hi+lo pairs, three fp16 MMAs per product: fp32-class (~22 bits per operand).
 *   FP16W : activations as fp16 hi+lo pairs, weights rounded once to fp16 (<= 2^-12 relative per weight), two MMAs per product.
 *   FP16  : the half-precision storage mode (= the reference's RGBA16F textures): one fp16 plane per tensor and per weight,
 *           one MMA per product, half the bytes. Meets the reference's half-precision tolerance (0.1,
 *           demo/common/testutil.h:1195), NOT the 1e-3 fp32 bar. */
enum { SNNB_PRECISION_FP32X3 = 0, SNNB_PRECISION_FP16W = 1, SNNB_PRECISION_FP16 = 2 };

/* ---- context / errors -------------------------------------------------------------------------------------- */
/* dp::BackendBuilder::build (core/src/ic2/backendBuilder.cpp:28-50) + context creation (core/src/contextFactory.cpp). */
int snnb_context_create(int device, snnb_context** out);
int snnb_context_destroy(snnb_context* ctx);
/* DeviceBackend::sync (backend.h:60; vulkanBackend.cpp:97-106 QueueSubmitAndWait). */
int snnb_sync(snnb_context* ctx);
/* The cudaStream_t everything is launched on (as void*). */
void* snnb_context_stream(snnb_context* ctx);
/* Thread-local message of the last failing call (replaces SNN_RIP / SNN_LOGE text, core/inc/snn/utils.h:57-62). */
const char* snnb_last_error(void);
/* Number of kernels this library has launched on the context since creation (bench.py's gpu_launches). */
uint64_t snnb_launch_count(snnb_context* ctx);
int snnb_version(void);
/* Default precision of per-operator convolution launches on this context (SNNB_PRECISION_FP32X3 or _FP16W; models carry
 * their own in snnb_model_options). */
int snnb_context_set_precision(snnb_context* ctx, int precision);

/* ---- tensors ------------------------------------------------------------------------------------------------ */
/* ImageTextureAllocator / ImageTexture::resetTexture + upload()/download() (imageTexture.h:60-147). */
int snnb_tensor_alloc(snnb_context* ctx, int n, int h, int w, int c, snnb_tensor** out);
int snnb_tensor_free(snnb_tensor* t);
int snnb_tensor_dims(const snnb_tensor* t, int* n, int* h, int* w, int* c);
int snnb_tensor_upload_nhwc(snnb_context* ctx, snnb_tensor* t, const float* host_nhwc);   /* synchronous */
int snnb_tensor_download_nhwc(snnb_context* ctx, const snnb_tensor* t, float* host_nhwc); /* synchronous */
/* Reference texture layout, per image: [ceil(C/4)][H][W][4]; images concatenated over N. */
int snnb_tensor_upload_c4hw4(snnb_context* ctx, snnb_tensor* t, const float* host_c4hw4);
int snnb_tensor_download_c4hw4(snnb_context* ctx, const snnb_tensor* t, float* host_c4hw4);
/* Debug dump in the reference's .dump format: 32-byte ASCII header "W H D C" + [D][H][W][4] fp32
 * (core/src/image.cpp:216-245). One file per image when N > 1 ("<path>.n<i>"). */
int snnb_tensor_dump(snnb_context* ctx, const snnb_tensor* t, const char* path);

/* ---- weights: fold + pack at load time ------------------------------------------------------------------------ */
/* Conv2DDesc (core/src/ic2/conv2d.h) + Conv2DLayer::getPaddingOffset (conv2d.cpp:39-74). pad_x/pad_y are the
 * shader's uPadx/uPady (NB the reference feeds offsets[0]=top as x and offsets[2]=left as y, conv2dVulkan.cpp:183-184). */
typedef struct {
    int in_channels, out_channels, kernel, stride;
    int pad_x, pad_y, pad_mode;
    int activation;
    float leaky_alpha;
    int algo; /* SNNB_ALGO_* */
} snnb_conv_desc;

/* Replaces Conv2DLayer::oihw2hwo4i4 (conv2d.cpp:76-100) + the BN/bias buffers of conv2dVulkan.cpp:110-152.
 * w_oihw: OC*IC*k*k (modelparser.cpp:641-657). bias / bn_* may be NULL. BN (eps 1e-3, sqrt clamp 1e-4,
 * vk_conv2d.comp:277-288) is folded into the packed weights and bias here. */
int snnb_weights_pack_conv2d(snnb_context* ctx, const snnb_conv_desc* d, const float* w_oihw, const float* bias, const float* bn_gamma,
                             const float* bn_beta, const float* bn_mean, const float* bn_var, snnb_weights** out);
/* Replaces SeparableConv2DLayer::oihw2hwo4i4 (separableconvolution.cpp:88-111). w_chw: C*k*k ([C][kh][kw], the
 * parser's mats, modelparser.cpp:827-850). in_channels == out_channels == C. */
int snnb_weights_pack_depthwise(snnb_context* ctx, const snnb_conv_desc* d, const float* w_chw, const float* bias, const float* bn_gamma,
                                const float* bn_beta, const float* bn_mean, const float* bn_var, snnb_weights** out);
/* Dense (denselayer.cpp:27-54): kernel is the flat JSON array viewed [out][in] (cpulayer.h:162). */
int snnb_weights_pack_dense(snnb_context* ctx, int n_in, int n_out, const float* kernel_out_in, const float* bias, snnb_weights** out);
/* Per-channel vectors (BatchNormalization: gamma,beta,mean,var; InstanceNorm: gamma,beta). Any may be NULL (defaults 1,0,0,1). */
int snnb_weights_pack_channels(snnb_context* ctx, int channels, const float* gamma, const float* beta, const float* mean, const float* var,
                               snnb_weights** out);
int snnb_weights_free(snnb_weights* w);

/* ---- operator launches (one call == one RenderPass::run, core/src/ic2/renderpass.h:64) ------------------------- */
/* Conv2D k x k incl. 1x1 (shadertemplate_vk_conv2d.comp:148-347, vk_conv2d_1x1.comp:68-211). `residual` (may be
 * NULL) is added before the activation: the fused form of Conv2D -> Add(+act) (vk_add.comp:41-90). */
int snnb_conv2d_launch(snnb_context* ctx, const snnb_conv_desc* d, const snnb_weights* w, const snnb_tensor* in, const snnb_tensor* residual,
                       snnb_tensor* out);
/* Depthwise k x k (shadertemplate_vk_depthwise.comp:64-139). */
int snnb_depthwise_launch(snnb_context* ctx, const snnb_conv_desc* d, const snnb_weights* w, const snnb_tensor* in, snnb_tensor* out);
/* MaxPooling2D / AveragePooling2D (vk_maxpool2d.comp:42-71, vk_avgpool2d.comp:42-69; window origin o*stride). */
int snnb_maxpool_launch(snnb_context* ctx, int kernel, int stride, const snnb_tensor* in, snnb_tensor* out);
int snnb_avgpool_launch(snnb_context* ctx, int kernel, int stride, const snnb_tensor* in, snnb_tensor* out);
/* Add + activation (vk_add.comp:41-90). */
int snnb_add_launch(snnb_context* ctx, int activation, float leaky_alpha, const snnb_tensor* a, const snnb_tensor* b, snnb_tensor* out);
/* Standalone BatchNormalization + activation (vk_batchnorm.comp:54-69); w from snnb_weights_pack_channels. */
int snnb_batchnorm_launch(snnb_context* ctx, const snnb_weights* w, int activation, float leaky_alpha, const snnb_tensor* in, snnb_tensor* out);
/* Standalone activation (vk_activation.comp:41-85). */
int snnb_activation_launch(snnb_context* ctx, int activation, float leaky_alpha, const snnb_tensor* in, snnb_tensor* out);
/* Dense + activation incl. softmax (cpulayer.h:136-261; GPU twin vk_dense.comp:53-83). in: [N,1,1,n_in] (or any
 * [N,H,W,C] with H*W*C == n_in, consumed in HWC order = CPU Flatten, cpulayer.h:94-115). out: [N,1,1,n_out]. */
int snnb_dense_launch(snnb_context* ctx, const snnb_weights* w, int activation, float leaky_alpha, const snnb_tensor* in, snnb_tensor* out);
/* Softmax over channels per pixel (cpulayer.h:175-191) and classifier index argmax+1 (core.cpp:228-233), per image. */
int snnb_softmax_launch(snnb_context* ctx, const snnb_tensor* in, snnb_tensor* out);
int snnb_argmax1(snnb_context* ctx, const snnb_tensor* in, int* host_idx_1based); /* synchronous; in: [N,1,1,C] */
/* Flatten in HWC order (cpulayer.h:94-115): [N,H,W,C] -> [N,1,1,H*W*C]. */
int snnb_flatten_launch(snnb_context* ctx, const snnb_tensor* in, snnb_tensor* out);
/* Concatenate along channels (vk_concat.comp:39-52). */
int snnb_concat_launch(snnb_context* ctx, const snnb_tensor* a, const snnb_tensor* b, snnb_tensor* out);
/* UpSampling2D nearest / bilinear (vk_upsampling2d_nearest.comp:43-64, _bilinear.comp:43-86). */
int snnb_upsample_launch(snnb_context* ctx, float scale, int bilinear, const snnb_tensor* in, snnb_tensor* out);
/* Pad constant/replicate/reflect (vk_pad.comp:42-70). */
int snnb_pad_launch(snnb_context* ctx, int pad_x, int pad_y, int pad_mode, const snnb_tensor* in, snnb_tensor* out);
/* InstanceNorm (+act), biased variance, eps 1e-5 (vk_instancenorm.comp:53-175). */
int snnb_instancenorm_launch(snnb_context* ctx, const snnb_weights* w, int activation, float leaky_alpha, const snnb_tensor* in, snnb_tensor* out);
/* Subpixel: depth_to_space(r) + tanh, always (vk_subpixel.comp:43-70, fs_subpixel.glsl:41). */
int snnb_subpixel_launch(snnb_context* ctx, int r, const snnb_tensor* in, snnb_tensor* out);

/* ---- device timers (DeviceBackend::createDeviceTimer, backend.h:79; core.cpp:140-152) --------------------------- */
int snnb_timer_create(snnb_context* ctx, snnb_timer** out);
int snnb_timer_start(snnb_timer* t);
int snnb_timer_stop(snnb_timer* t);
int snnb_timer_elapsed_ms(snnb_timer* t, float* ms); /* synchronises on the stop event */
int snnb_timer_destroy(snnb_timer* t);

/* ---- launch capture for backend-level integration -------------------------------------------------------------
 * A DeviceBackend built on the per-operator calls (INTEGRATION.md, depth B) records its stage loop once and replays it:
 * everything launched on the context between capture_begin and capture_end becomes one CUDA graph (the counterpart of
 * recording the reference's single command buffer, vulkanBackend.cpp:97-106). Run the same launches eagerly once before
 * capturing: lazily created resources (tensor-map encoder, split-K scratch) must exist, because allocation is illegal
 * while capturing. Tensors and weights referenced by the graph must outlive it. */
typedef struct snnb_graph snnb_graph;
int snnb_graph_capture_begin(snnb_context* ctx);
int snnb_graph_capture_end(snnb_context* ctx, snnb_graph** out);
int snnb_graph_launch(snnb_graph* g); /* asynchronous on the context's stream */
int snnb_graph_destroy(snnb_graph* g);

/* ---- whole-model engine: dp::loadFromJsonModel + generateInferenceGraph + MixedInferenceCore ------------------- */
typedef struct {
    int batch;          /* images per run() on this GPU (the reference is fixed at 1, inferencegraph.h:58-64) */
    int input_width;    /* ShaderGenOptions::desiredInput (layeroption.h:30); 0 = use the JSON InputLayer's */
    int input_height;
    int conv_algo;      /* SNNB_ALGO_*: AUTO by default */
    int use_cuda_graph; /* replay the captured forward pass instead of re-launching kernels */
    int fuse;           /* graph-level fusion passes (conv+add+act, pad->conv); 0 keeps 1 kernel per reference layer */
    int precision;      /* SNNB_PRECISION_*; FP16 = the reference's preferrHalfPrecision (layeroption.h:43) */
} snnb_model_options;

/* MixedInferenceCore::create(ctx, modelFileName, options) (core.h:115-116) = dp::loadFromJsonModel (dp.cpp:115-167:
 * ModelParser ctor modelparser.cpp:210-258 incl. the sidecar .bin next to the JSON) + generateInferenceGraph
 * (dp.cpp:432-640) + init (core.cpp:294-410) + weight fold/pack/upload. */
int snnb_model_load_json(snnb_context* ctx, const char* json_path, const snnb_model_options* opt, snnb_model** out);
int snnb_model_destroy(snnb_model* m);
int snnb_model_num_layers(const snnb_model* m);
/* Layer i in JSON order: name "<json file> layer [NN] <Type>" (dp.cpp:135), type string, output dims. */
int snnb_model_layer_info(const snnb_model* m, int i, char* name, int name_cap, char* type, int type_cap, int* n, int* h, int* w, int* c);
int snnb_model_num_inputs(const snnb_model* m);
int snnb_model_num_outputs(const snnb_model* m);
int snnb_model_input_dims(const snnb_model* m, int idx, int* n, int* h, int* w, int* c);
int snnb_model_output_dims(const snnb_model* m, int idx, int* n, int* h, int* w, int* c);
/* MixedInferenceCore::run (core.cpp:97-245), end to end with HOST buffers: H2D of the NHWC fp32 batch, forward,
 * D2H of output 0 (NHWC fp32, out_capacity floats) and, for classifiers (last layer Dense/softmax), the 1-based
 * class index per image (core.cpp:228-233); classes may be NULL. Synchronous. */
int snnb_model_run(snnb_model* m, const float* host_input_nhwc, float* host_output, size_t out_capacity, int* classes_1based);
/* Streaming variant of snnb_model_run for serving loops: submit() enqueues the H2D copy of the batch (on a dedicated copy
 * stream, double-buffered device staging), the forward pass and the D2H copies of output 0 / class indices into the
 * caller's buffers, and returns at once with a ticket; wait(ticket) blocks until that submission's results are in host
 * memory. Up to two submissions may be in flight, so batch i+1's upload overlaps batch i's compute. Host buffers must be
 * pinned for the copies to be asynchronous and must stay untouched until wait() returns. (The reference's run() is
 * strictly synchronous, core.cpp:97-245; this is additive.) */
int snnb_model_submit(snnb_model* m, const float* host_input_nhwc, float* host_output, size_t out_capacity, int* classes_1based, int* ticket);
/* submit() for 8-bit images: host_input is N*H*W*C bytes (NHWC, dense); the device computes (x - mean4[c & 3]) * norm4[c & 3]
 * while converting, i.e. ImageTexture::convertToRGBA32FAndNormalize(means, norms) (core/inc/snn/imageTexture.h:114; per-model
 * constants in demo/common/modelInference.cpp:135-224, e.g. ResNet-18 mean 127.5 norm 1/127.5) without a host pass, and a
 * quarter of the fp32 bytes cross PCIe. */
int snnb_model_submit_u8(snnb_model* m, const uint8_t* host_input_nhwc_u8, const float* mean4, const float* norm4, float* host_output, size_t out_capacity,
                         int* classes_1based, int* ticket);
/* Image in, image (or tensor) out, all pre/post-processing on the device (SURVEY §8 f-N3): the 8-bit input may have ANY size - it is
 * resized to the model's input with the linear or nearest filter exactly as ImageTexture::resize does (imageTexture.h:137,
 * shadertemplate_vk_resize.comp:42-61: output texel centres sampled from the source) and normalised in the same kernel; the result comes
 * back either as fp32 (output_f32) or as an 8-bit image, clamp(round(v * out_scale + out_offset), 0, 255) (style transfer: scale 1;
 * a tanh output: 127.5 / 127.5). Same ticket / wait protocol as snnb_model_submit. */
typedef struct {
    const uint8_t* input_u8; /* N * src_height * src_width * C bytes, NHWC, dense */
    int src_height, src_width;
    int linear_filter;       /* 1 = linear (the reference's default), 0 = nearest */
    float mean4[4], norm4[4];
    float* output_f32;       /* exactly one of output_f32 / output_u8 may be non-NULL (both NULL: no output copy) */
    size_t output_capacity;  /* elements */
    uint8_t* output_u8;
    float out_scale, out_offset;
    int* classes_1based;     /* classifiers only, may be NULL */
} snnb_image_io;
int snnb_model_submit_image(snnb_model* m, const snnb_image_io* io, int* ticket);
int snnb_model_wait(snnb_model* m, int ticket);
/* Device-resident variant: inputs already uploaded with snnb_model_set_input(); forward only, asynchronous. */
int snnb_model_set_input(snnb_model* m, int idx, const float* host_input_nhwc);
int snnb_model_forward(snnb_model* m);
int snnb_model_get_output(snnb_model* m, int idx, float* host_output, size_t out_capacity);
/* Output of any layer (JSON index) as host NHWC fp32 — the per-layer checkpoint the reference's model tests compare
 * (demo/test/unittest/resnet18Test.cpp:85-198). Requires that the layer was not fused away (fuse=0) . */
int snnb_model_layer_output(snnb_model* m, int layer, float* host_nhwc, size_t capacity);
/* Dump every layer's output as "<dir>/<name> pass[0].dump" (vulkanBackend.cpp:108-143). */
int snnb_model_dump_outputs(snnb_model* m, const char* dir);
/* Per-layer device time of one forward pass, ms, via event pairs (writeTimeStat, core.cpp:437-442). times[num_layers]. */
int snnb_model_time_layers(snnb_model* m, float* times_ms, int capacity);
/* Name of the CUDA kernel layer `layer` launched in the last snnb_model_time_layers() pass ("" for a layer that launched none:
 * inputs, fused-away layers). What bench.py attributes the per-kernel roofline to. */
int snnb_model_layer_kernel(const snnb_model* m, int layer, char* name, int name_cap);
/* Kernels launched by one forward pass. */
int snnb_model_launches_per_forward(const snnb_model* m);
/* YOLO detection output of the last run (yololayer.cpp:177-226): rows {class, score, x, y, w, h}; returns the
 * number of boxes for image `n` via *count. */
int snnb_model_get_boxes(snnb_model* m, int n, float* rows6, int max_rows, int* count);
/* The packed weight arena (device pointer, bytes): rank 0 packs, the caller broadcasts it once with NCCL
 * (torch.distributed) and no collective ever runs on the forward path (SURVEY §8e). */
int snnb_model_weight_arena(snnb_model* m, void** device_ptr, size_t* bytes);

/* ---- multi-GPU: the ONE collective of the engine, in C++ (SURVEY §8b/e) --------------------------------------------
 * One process per GPU. Rank `root` packs the weights; every other rank receives the packed arena with a single ncclBroadcast
 * on the context's stream. NCCL is resolved at run time (the process's already-loaded libnccl.so.2 - e.g. PyTorch's - else
 * dlopen): the library has no link-time dependency on it. Bootstrap: rank 0 calls snnb_nccl_unique_id and ships the 128
 * bytes to the others by whatever means the host has (MPI, a file, torch.distributed), then every rank creates its
 * communicator. No collective ever runs on the forward path. (The reference is single-device: new surface, kept thin.) */
typedef struct snnb_comm snnb_comm;
int snnb_nccl_unique_id(unsigned char id128[128]);
int snnb_nccl_comm_create(snnb_context* ctx, int rank, int world_size, const unsigned char id128[128], snnb_comm** out);
int snnb_nccl_comm_destroy(snnb_comm* comm);
int snnb_bcast_weights(snnb_model* m, snnb_comm* comm, int root); /* asynchronous on the context's stream */

/* ---- layer registration: snn::dp::registerLayer(name, LayerCreator) (core/src/ic2/layerFactory.h:116-122) ------------
 * A host registers a creator for a layer `type` string; when a model file names that type, the creator is called with a
 * read-only view of the "Layer_<i>" JSON object (the accessors below = what ModelParser hands the reference's creators,
 * modelparser.h:60-157) and fills in the implementation: how the output dims follow from the inputs' and what to launch.
 * `run` works on the context's stream with this header's own operator launches (or its own kernels on the tensors' planes).
 * Registering an existing name replaces it, as registerLayer() does (built-in types included). */
typedef struct snnb_layer_json snnb_layer_json;
int snnb_layer_json_number(const snnb_layer_json* layer, const char* key, double* out);             /* 0 = present and numeric */
int snnb_layer_json_string(const snnb_layer_json* layer, const char* key, char* buf, int cap);      /* 0 = present and a string */
/* numeric array at a dotted path ("weights.kernel"); the pointer stays valid during the creator call only */
int snnb_layer_json_numbers(const snnb_layer_json* layer, const char* path, const double** data, size_t* count);
typedef struct {
    void* user;
    /* hwc triples: in_hwc[3*i .. 3*i+2] = (height, width, channels) of input i; write the output's into out_hwc[3]. 0 = ok. */
    int (*output_dims)(void* user, int num_inputs, const int* in_hwc, int* out_hwc);
    /* enqueue the layer's work on snnb_context_stream(ctx). 0 = ok. */
    int (*run)(void* user, snnb_context* ctx, int num_inputs, const snnb_tensor* const* inputs, snnb_tensor* output);
    void (*destroy)(void* user); /* may be NULL */
} snnb_layer_impl;
typedef int (*snnb_layer_creator)(void* registry_user, const snnb_layer_json* layer, snnb_layer_impl* out);
int snnb_register_layer(const char* type_name, snnb_layer_creator creator, void* registry_user);
int snnb_unregister_layer(const char* type_name);
/* Raw device planes of a tensor for custom kernels: NHWC, channel pitch `cp` (a multiple of 8), fp16 hi plane and lo plane
 * (value = hi + lo; lo is NULL in the half-precision storage mode). */
int snnb_tensor_planes(const snnb_tensor* t, void** hi, void** lo, int* cp);
/* Diagnostics: the work decomposition SNNB_ALGO_TCGEN05_STREAMK would use for `tiles` output tiles of `num_kb` K blocks on `sms` SMs,
 * evaluated on the host with the kernel's own arithmetic. rows = capacity x 6 ints {cta, tile, kb0, kb1, piece, pieces} in each CTA's
 * order; returns the number of rows (may exceed capacity), -1 when the tile count is a multiple of `sms` or too small to cut. No GPU needed. */
int snnb_debug_streamk_schedule(int tiles, int num_kb, int sms, int* rows, int capacity);
/* Diagnostics: the K layout of the stem kernel's feed mode for a k x k stride-`stride` convolution with `ic` input channels and x padding
 * `pad_x`: out = {px (left margin of the compact input copy), d (pixel offset of tap 0 in the window), nch (16-byte chunks per window),
 * ksteps (K = 16 steps per filter row), rows_per_panel (filter rows sharing one 128-byte weight row)}. Returns 1 if the layer can use
 * the feed mode, 0 if not. No GPU needed. */
int snnb_debug_feed_plan(int k, int stride, int pad_x, int ic, int out[5]);
/* Diagnostics: every K block the tensor-core producer loads for a `ksize` x `ksize` convolution over `cblocks` 64-channel blocks (channel
 * pitch `icp`) with a folded 1x1 shortcut of `sc_cblocks` channel blocks (0: none), for `tiles` output tiles split into `ksplit` K ranges
 * (0: stream-K over `sms` SMs). rows = capacity x 6 ints {tile, kb, shortcut, tap, channel block, weight column}, in each work item's
 * order; returns the number of rows (may exceed capacity), -1 for invalid arguments or nothing to cut (stream-K). No GPU needed. */
int snnb_debug_kblock_schedule(int ksize, int cblocks, int icp, int sc_cblocks, int tiles, int ksplit, int sms, int* rows, int capacity);

#ifdef __cplusplus
}
#endif
#endif /* SNNB_H_ */
