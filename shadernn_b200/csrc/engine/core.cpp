// MixedInferenceCore: init (tensor plan, weight arena, fusion, CUDA-graph capture) and run.
// Counterpart of core/src/ic2/core.cpp:294-410 (init) and :97-245 (run).
#include <algorithm>
#include <cstring>
#include <unordered_map>
#include <unordered_set>

#include "engine.h"

using namespace snnb;

namespace snn {

using namespace dp;

MixedInferenceCore::~MixedInferenceCore() {
    if (ctx) {
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
    }
    if (cuGraphExec) cudaGraphExecDestroy(cuGraphExec);
    if (cuGraph) cudaGraphDestroy(cuGraph);
    for (auto* t : ownedTensors) snnb_tensor_free(t);
    if (arena) cudaFree(arena);
    if (scratchArena) cudaFree(scratchArena);
    if (ioStage) cudaFree(ioStage);
    if (argmaxDev) cudaFree(argmaxDev);
    if (yoloDev) cudaFree(yoloDev);
    if (yoloHost) cudaFreeHost(yoloHost);
    for (auto& sl : slots) {
        if (sl.yoloDev) cudaFree(sl.yoloDev);
        if (sl.yoloHost) cudaFreeHost(sl.yoloHost);
        if (sl.stageIn) cudaFree(sl.stageIn);
        if (sl.stageResize) cudaFree(sl.stageResize);
        if (sl.stageOut) cudaFree(sl.stageOut);
        if (sl.smallHost) cudaFreeHost(sl.smallHost);
        if (sl.argmax) cudaFree(sl.argmax);
        if (sl.h2dDone) cudaEventDestroy(sl.h2dDone);
        if (sl.stageFree) cudaEventDestroy(sl.stageFree);
        if (sl.resultReady) cudaEventDestroy(sl.resultReady);
    }
    if (copyStream) cudaStreamDestroy(copyStream);
}

std::unique_ptr<MixedInferenceCore> MixedInferenceCore::create(snnb_context* ctx, const std::string& modelFileName, const ShaderGenOptions& options,
                                                               std::string& err) {
    std::unique_ptr<MixedInferenceCore> core(new MixedInferenceCore());
    core->ctx     = ctx;
    core->options = options;
    try {
        core->layers = loadFromJsonModel(modelFileName);
        core->graph  = generateInferenceGraph(core->layers, options);
    } catch (std::exception& e) {
        err = e.what();
        return nullptr;
    }
    if (!core->init(err)) return nullptr;
    return core;
}

static bool allZeroPadding(const PaddingSpec& p) {
    uint32_t o[4];
    p.offsets(3, true, o); // kernel size only matters for "same"
    const bool keyword_same = !(p.t == "valid" || p.t == "none" || (!p.t.empty() && std::all_of(p.t.begin(), p.t.end(), ::isdigit)));
    return !keyword_same && o[0] == 0 && o[1] == 0 && o[2] == 0 && o[3] == 0;
}

bool MixedInferenceCore::init(std::string& err) {
    const int N = (int) options.batch;
    // ShaderGenOptions::preferrHalfPrecision (layeroption.h:43 -> RGBA16F textures): every tensor is ONE fp16 plane
    const bool twoPlanes = options.precision != SNNB_PRECISION_FP16;
    std::unordered_map<GenericModelLayer*, int> order;
    for (size_t i = 0; i < graph.sorted.size(); ++i) order[graph.sorted[i]] = (int) i;

    for (auto* L : graph.sorted) {
        if (L->isInputLayer) inputLayers.push_back(L);
        if (L->nextLayers.empty()) outputLayers.push_back(L);
        if (L->typeName == "YOLO") yolo = static_cast<YOLOLayer*>(L);
    }
    std::stable_sort(inputLayers.begin(), inputLayers.end(), [](GenericModelLayer* a, GenericModelLayer* b) {
        return static_cast<InputLayerLayer*>(a)->_desc.inputIndex < static_cast<InputLayerLayer*>(b)->_desc.inputIndex;
    });
    if (inputLayers.empty()) {
        err = "model has no InputLayer";
        return false;
    }

    // ---- fusion passes (engine-level; off => one kernel per reference layer, every layer output observable) ----
    // `alias[L]` = the layer whose output tensor stands in for L's (L launches nothing).
    std::unordered_map<GenericModelLayer*, GenericModelLayer*> alias;
    // SNNB_NO_SHORTCUT_FOLD: profiling switch, read at every load so that one process can compare both forms
    const bool shortcutFold = options.fuse && options.convAlgo != SNNB_ALGO_SIMT && getenv("SNNB_NO_SHORTCUT_FOLD") == nullptr;
    // Can `c2` (k x k, stride 1) take the 1x1 projection `ds` of another tensor as extra K blocks? Shapes, order and the tensor-core
    // planner decide (conv2d_umma_fold_supported, asked with stand-in tensors of the planned shapes: nothing is allocated yet).
    auto foldable = [&](GenericModelLayer* c2, GenericModelLayer* ds) {
        if (c2 == ds || c2->typeName != "Conv2D" || ds->typeName != "Conv2D" || c2->fusedAway || ds->fusedAway) return false;
        auto* cc = static_cast<Conv2DLayer*>(c2);
        auto* dc = static_cast<Conv2DLayer*>(ds);
        if (c2->nextLayers.size() != 1 || ds->nextLayers.size() != 1 || c2->prevLayers.size() != 1 || ds->prevLayers.size() != 1) return false;
        if (cc->_desc.activation.id != SNNB_ACT_NONE || dc->_desc.activation.id != SNNB_ACT_NONE || cc->residual || cc->fusedAct >= 0 || cc->shortcut ||
            dc->shortcut || dc->foldedInto)
            return false;
        // a 1x1 convolution runs with pad 0 whatever its padding spec says (Conv2DLayer::run): the fold reads what its own launch reads
        const int dsMode = padModeId(dc->_desc.padding.mode);
        if (cc->_desc.stride != 1 || dc->_desc.kernelSize != 1 || !(dsMode == SNNB_PAD_NONE || dsMode == SNNB_PAD_CONSTANT)) return false;
        GenericModelLayer* x = ds->prevLayers[0];
        if (order[x] >= order[c2]) return false; // the shortcut's input must be complete when c2 runs
        const Dims &dc2 = graph.outputDims[order[c2]], &dds = graph.outputDims[order[ds]];
        if (dc2.width != dds.width || dc2.height != dds.height || dc2.depth != dds.depth || graph.outputDims[order[x]].depth != ds->numInputPlanes) return false;
        auto stand_in = [&](GenericModelLayer* X) {
            snnb_tensor t;
            const Dims& d = graph.outputDims[order[X]];
            t.n = N, t.h = (int) d.height, t.w = (int) d.width, t.c = (int) d.depth, t.cp = round_up(t.c, 8);
            t.hi = reinterpret_cast<__half*>(1), t.lo = twoPlanes ? t.hi : nullptr;
            return t;
        };
        const snnb_tensor in = stand_in(c2->prevLayers[0]), sc = stand_in(x), out = stand_in(c2);
        snnb_weights probe; // "tensor path available", with the row-window operand the layer would be packed with (as wantsPrepad asks)
        probe.w_hi = probe.w_lo = probe.w_row_hi = probe.w_row_lo = reinterpret_cast<__half*>(1);
        uint32_t offs[4];
        cc->_desc.padding.offsets((int) cc->_desc.kernelSize, true, offs);
        ConvArgs a;
        a.in = &in, a.residual = nullptr, a.out = const_cast<snnb_tensor*>(&out), a.w = &probe;
        a.k = (int) cc->_desc.kernelSize, a.stride = 1;
        a.pad_x = a.k == 1 ? 0 : (int) offs[0], a.pad_y = a.k == 1 ? 0 : (int) offs[2], a.pad_mode = padModeId(cc->_desc.padding.mode);
        probe.row_stride = 1, probe.row_pad = a.pad_x;
        a.act = SNNB_ACT_NONE, a.alpha = 0.0f, a.precision = options.precision;
        a.shortcut = &sc, a.sc_stride = (int) dc->_desc.stride;
        return conv2d_umma_fold_supported(ctx, a);
    };
    if (options.fuse) {
        for (auto* L : graph.sorted) {
            // (1) Pad -> Conv2D/Depthwise with zero own padding: the consumer's gather applies the offsets (and mode) itself.
            if (L->typeName == "Pad" && L->nextLayers.size() == 1 && L->prevLayers.size() == 1) {
                auto* pad  = static_cast<PadLayer*>(L);
                auto* next = L->nextLayers[0];
                PaddingSpec* np = nullptr;
                if (next->typeName == "Conv2D" && static_cast<Conv2DLayer*>(next)->_desc.kernelSize > 1) np = &static_cast<Conv2DLayer*>(next)->_desc.padding;
                if (next->typeName == "SeparableConv2D" && pad->mode == "constant") np = &static_cast<SeparableConv2DLayer*>(next)->_desc.padding;
                if (np && allZeroPadding(*np)) {
                    uint32_t o[4];
                    pad->padding.offsets(0, false, o);
                    np->t = std::to_string(o[0]), np->b = std::to_string(o[1]), np->l = std::to_string(o[2]), np->r = std::to_string(o[3]);
                    np->mode       = pad->mode;
                    L->fusedAway   = true;
                    alias[L]       = L->prevLayers[0];
                }
            }
            // (5) Conv2D(k x k, stride 1) + Conv2D(1x1 projection of another tensor) -> Add(+act), as in a down-sampling ResNet block:
            // Add(c2(y), ds(x)) = [W2 | Wds] . [im2col(y) ; x_strided] + (b2 + bds), one GEMM whose K loop runs on into the projection's
            // channels. c2 writes the Add's tensor with the Add's activation; ds and the Add launch nothing, and ds has no tensor.
            // Where it cannot fire, (2) fuses the Add into one of the convs as before.
            if (shortcutFold && L->typeName == "Add" && L->prevLayers.size() == 2) {
                auto* add = static_cast<AddLayer*>(L);
                for (int o = 0; o < 2; ++o) {
                    GenericModelLayer* c2 = L->prevLayers[o];
                    GenericModelLayer* ds = L->prevLayers[1 - o];
                    if (!foldable(c2, ds)) continue;
                    auto* cc       = static_cast<Conv2DLayer*>(c2);
                    cc->fusedAct   = add->activation.id;
                    cc->fusedAlpha = add->activation.alpha;
                    cc->shortcut   = static_cast<Conv2DLayer*>(ds);
                    cc->shortcut->foldedInto = cc;
                    ds->fusedAway  = true;
                    L->fusedAway   = true;
                    alias[c2]      = L; // c2 output == add output
                    break;
                }
            }
            // (2) Conv2D(linear) -> Add(+act): the conv's epilogue adds the other operand and applies the Add's activation.
            if (L->typeName == "Add" && L->prevLayers.size() == 2 && !L->fusedAway) {
                auto* add = static_cast<AddLayer*>(L);
                GenericModelLayer* a = L->prevLayers[0];
                GenericModelLayer* b = L->prevLayers[1];
                auto fusable = [&](GenericModelLayer* c, GenericModelLayer* other) {
                    if (c->typeName != "Conv2D" || c->nextLayers.size() != 1 || c->fusedAway) return false;
                    auto* conv = static_cast<Conv2DLayer*>(c);
                    if (conv->_desc.activation.id != SNNB_ACT_NONE || conv->residual || conv->fusedAct >= 0) return false;
                    return order[other] < order[c] && c != other; // the other operand must be complete before the conv runs
                };
                GenericModelLayer* conv = nullptr;
                GenericModelLayer* other = nullptr;
                if (fusable(b, a))
                    conv = b, other = a;
                else if (fusable(a, b))
                    conv = a, other = b;
                if (conv) {
                    conv->fusedAct   = add->activation.id;
                    conv->fusedAlpha = add->activation.alpha;
                    conv->prevLayers.push_back(other); // bookkeeping only: residual operand
                    L->fusedAway     = true;           // the Add launches nothing; its tensor is written by the conv
                    alias[conv]      = L;              // conv output == add output
                }
            }
            // (4) global AveragePooling2D -> [Flatten] -> Dense with few units: one classifier-head launch (gap_dense_kernel).
            if (L->typeName == "Dense" && L->prevLayers.size() == 1) {
                GenericModelLayer* f = L->prevLayers[0];
                GenericModelLayer* pool = (f->typeName == "Flatten" && f->prevLayers.size() == 1 && f->nextLayers.size() == 1 &&
                                           static_cast<FlattenLayer*>(f)->activation.id == SNNB_ACT_NONE)
                                              ? f->prevLayers[0]
                                              : f;
                auto dimsOf = [&](GenericModelLayer* x) { return graph.outputDims[order[x]]; };
                if (pool->typeName == "AveragePooling2D" && static_cast<PoolingLayer*>(pool)->isAvg && pool->nextLayers.size() == 1 && pool->prevLayers.size() == 1 &&
                    !pool->fusedAway && dimsOf(pool).width * dimsOf(pool).height == 1 && static_cast<DenseLayer*>(L)->units <= 256 &&
                    dimsOf(pool->prevLayers[0]).width * dimsOf(pool->prevLayers[0]).height >= 4 && dimsOf(pool->prevLayers[0]).depth <= 4096 &&
                    static_cast<PoolingLayer*>(pool)->_desc.kernelSize >= dimsOf(pool->prevLayers[0]).width &&
                    static_cast<PoolingLayer*>(pool)->_desc.kernelSize >= dimsOf(pool->prevLayers[0]).height) {
                    static_cast<DenseLayer*>(L)->gapSource = pool->prevLayers[0];
                    pool->fusedAway = true; // launches nothing; keeps its own (unwritten) 1x1 tensor so that shapes downstream still check
                }
            }
            // (3) Flatten of a 1x1xC tensor without activation is the identity.
            if (L->typeName == "Flatten" && L->inputDims.size() == 1 && L->inputDims[0].width * L->inputDims[0].height == 1 &&
                static_cast<FlattenLayer*>(L)->activation.id == SNNB_ACT_NONE) {
                L->fusedAway = true;
                alias[L]     = L->prevLayers[0];
            }
        }
    }

    // ---- tensors: one output per executing layer (core.cpp:356-374 allocates one texture per stage) ----
    std::unordered_map<GenericModelLayer*, snnb_tensor*> outOf;
    auto resolve = [&](GenericModelLayer* L) -> GenericModelLayer* {
        std::unordered_set<GenericModelLayer*> seen;
        while (alias.count(L) && !seen.count(L)) {
            seen.insert(L);
            L = alias[L];
        }
        return L;
    };
    for (size_t i = 0; i < graph.sorted.size(); ++i) {
        GenericModelLayer* L = graph.sorted[i];
        if (L->typeName == "YOLO") continue; // host op
        GenericModelLayer* owner = resolve(L);
        if (owner != L && !(L->typeName == "Conv2D")) continue; // Pad/Flatten aliases own nothing
        if (L->typeName == "Conv2D" && static_cast<Conv2DLayer*>(L)->foldedInto) continue; // a folded shortcut writes nothing
        if (outOf.count(owner)) continue;
        // dims of the tensor = dims of `owner` (for conv->add fusion both agree)
        const Dims& d = graph.outputDims[order[owner]];
        snnb_tensor* t = nullptr;
        if (tensor_alloc(ctx, N, (int) d.height, (int) d.width, (int) d.depth, &t, twoPlanes)) {
            err = get_error();
            return false;
        }
        ownedTensors.push_back(t);
        outOf[owner] = t;
    }
    for (auto* L : graph.sorted) {
        if (L->typeName == "YOLO") {
            for (auto* p : L->prevLayers) L->inputs.push_back(outOf.at(resolve(p)));
            continue;
        }
        GenericModelLayer* owner = resolve(L);
        L->output                = outOf.count(owner) ? outOf[owner] : nullptr;
        if (L->fusedAway) continue;
        size_t nin = L->prevLayers.size();
        if (L->typeName == "Conv2D" && static_cast<Conv2DLayer*>(L)->fusedAct >= 0 && !static_cast<Conv2DLayer*>(L)->shortcut) {
            nin -= 1; // last prev is the residual operand
            L->residual = outOf.at(resolve(L->prevLayers.back()));
        }
        for (size_t k = 0; k < nin; ++k) L->inputs.push_back(outOf.at(resolve(L->prevLayers[k])));
        if (L->typeName == "Conv2D") {
            auto* cl  = static_cast<Conv2DLayer*>(L);
            cl->algo = options.convAlgo;
            if (cl->shortcut) cl->shortcutIn = outOf.at(resolve(cl->shortcut->prevLayers[0]));
            // weights are not packed yet: probe with a weights stub that says "tensor path available"
            int ph = 0, pw = 0;
            snnb_weights probe_w;
            probe_w.w_hi = probe_w.w_lo = reinterpret_cast<__half*>(1);
            // ... and the row-window operand a pre-padded small-channel stem will be packed with (stride, pad 0; packWeights)
            probe_w.w_row_hi = probe_w.w_row_lo = reinterpret_cast<__half*>(1);
            probe_w.row_stride = (int) cl->_desc.stride, probe_w.row_pad = 0;
            std::swap(cl->weights, probe_w);
            const bool prepad = cl->wantsPrepad(L->inputs[0], L->output, options.convAlgo, ph, pw);
            std::swap(cl->weights, probe_w);
            if (prepad) {
                if (tensor_alloc(ctx, N, ph, pw, L->inputs[0]->c, &cl->prepadded, twoPlanes)) {
                    err = get_error();
                    return false;
                }
                ownedTensors.push_back(cl->prepadded);
            }
            // a stride-2 RGB stem fed straight by a model input: give that input tensor the compact 4-channel copy (feed mode)
            {
                static const bool noFeed = getenv("SNNB_NO_FEED") != nullptr;
                GenericModelLayer* src   = resolve(L->prevLayers[0]);
                snnb_tensor* in          = L->inputs[0];
                const int mode           = padModeId(cl->_desc.padding.mode);
                uint32_t offs[4];
                cl->_desc.padding.offsets((int) cl->_desc.kernelSize, true, offs);
                const int k = (int) cl->_desc.kernelSize, padX = (int) offs[0], padY = (int) offs[2];
                FeedPlan fp;
                if (!noFeed && !prepad && src->isInputLayer && !in->feed_hi && options.convAlgo != SNNB_ALGO_SIMT && !L->residual && !cl->shortcut && L->output->c <= 64 &&
                    (mode == SNNB_PAD_NONE || mode == SNNB_PAD_CONSTANT) && make_feed_plan(k, (int) cl->_desc.stride, padX, in->c, fp)) {
                    const int tilesX = (L->output->w + 127) / 128;
                    const int needW  = 2 * (tilesX * 128 - 1) + 2 * fp.nch;          // last pixel a tile's window segment touches + 1
                    const int needH  = 2 * (L->output->h - 1) + k - padY + padY;      // last input row + 1, shifted by feed_py = padY
                    const int feedW  = (std::max(in->w + fp.px, needW) + 1) & ~1;
                    const int feedH  = std::max(in->h + padY, needH);
                    if (tensor_alloc_feed(in, feedH, feedW, padY, fp.px)) {
                        err = get_error();
                        return false;
                    }
                    cl->feedInput = true;
                }
            }
        }
        if (L->typeName == "Dense") {
            auto* dl = static_cast<DenseLayer*>(L);
            if (L->inputs[0]->h * L->inputs[0]->w != 1) {
                if (tensor_alloc(ctx, N, 1, 1, (int) dl->numInputPlanes, &dl->flat, twoPlanes)) {
                    err = get_error();
                    return false;
                }
                ownedTensors.push_back(dl->flat);
            }
            if ((uint32_t) (L->inputs[0]->h * L->inputs[0]->w * L->inputs[0]->c) != dl->numInputPlanes) {
                err = L->name + ": Dense expects " + std::to_string(dl->numInputPlanes) + " inputs, graph provides " +
                      std::to_string(L->inputs[0]->h * L->inputs[0]->w * L->inputs[0]->c);
                return false;
            }
        }
        if ((L->typeName == "Add" || L->typeName == "Concatenate") && L->inputs.size() != 2) {
            err = L->name + ": expects exactly two inputs";
            return false;
        }
        // The kernels index weights and operands with the RUNTIME tensors' extents: a model whose declared planes disagree with
        // what the graph produces would read out of bounds on the device. Reject it here, as a load error.
        auto dimsStr = [](const snnb_tensor* t) { return std::to_string(t->h) + "x" + std::to_string(t->w) + "x" + std::to_string(t->c); };
        if (L->typeName == "Conv2D" || L->typeName == "SeparableConv2D" || L->typeName == "BatchNormalization" || L->typeName == "InstanceNorm") {
            if (L->inputs.empty() || !L->output) {
                err = L->name + ": layer has no input";
                return false;
            }
            if ((uint32_t) L->inputs[0]->c != L->numInputPlanes) {
                err = L->name + ": inputPlanes " + std::to_string(L->numInputPlanes) + " but the producing layer has " + std::to_string(L->inputs[0]->c) + " channels";
                return false;
            }
            const uint32_t wantOut = (L->typeName == "Conv2D") ? L->numOutputPlanes : L->numInputPlanes;
            if ((uint32_t) L->output->c != wantOut) {
                err = L->name + ": output tensor has " + std::to_string(L->output->c) + " channels, weights are packed for " + std::to_string(wantOut);
                return false;
            }
        }
        if (L->typeName == "Add") {
            for (auto* in : L->inputs)
                if (in->h != L->output->h || in->w != L->output->w || in->c != L->output->c) {
                    err = L->name + ": Add operand " + dimsStr(in) + " does not match the output " + dimsStr(L->output);
                    return false;
                }
        }
        if (L->typeName == "Conv2D" && L->residual &&
            (L->residual->h != L->output->h || L->residual->w != L->output->w || L->residual->c != L->output->c)) {
            err = L->name + ": fused Add operand " + dimsStr(L->residual) + " does not match the output " + dimsStr(L->output);
            return false;
        }
        if (L->typeName == "Concatenate") {
            if (L->inputs[0]->h != L->inputs[1]->h || L->inputs[0]->w != L->inputs[1]->w || L->inputs[0]->c + L->inputs[1]->c != L->output->c ||
                L->inputs[0]->h != L->output->h || L->inputs[0]->w != L->output->w) {
                err = L->name + ": Concatenate operands " + dimsStr(L->inputs[0]) + " and " + dimsStr(L->inputs[1]) + " do not stack into " + dimsStr(L->output);
                return false;
            }
        }
    }

    // input tensors whose ONLY readers are feed-mode stems need no regular planes (snnb_tensor::feed_only)
    for (auto* in : inputLayers) {
        snnb_tensor* t = in->output;
        if (!t || !t->feed_hi || getenv("SNNB_NO_FEED_ONLY")) continue;
        bool only = true;
        int readers = 0;
        for (auto* L : graph.sorted) {
            if (L->fusedAway || L->isInputLayer) continue;
            const bool reads = std::find(L->inputs.begin(), L->inputs.end(), t) != L->inputs.end() || L->residual == t ||
                               (L->typeName == "Conv2D" && static_cast<Conv2DLayer*>(L)->shortcutIn == t);
            if (!reads) continue;
            ++readers;
            only = only && L->typeName == "Conv2D" && static_cast<Conv2DLayer*>(L)->feedInput && L->inputs.size() >= 1 && L->inputs[0] == t && L->residual != t &&
                   std::count(L->inputs.begin(), L->inputs.end(), t) == 1;
        }
        for (auto* o : outputLayers) only = only && o->output != t; // a model that returns its input
        t->feed_only = only && readers > 0;
    }

    // ---- weights: fold + pack on the host, then ONE device arena (broadcastable with a single NCCL call) ----
    std::vector<std::pair<GenericModelLayer*, PackedHost>> packed;
    size_t total = 0, scratchTotal = 0;
    for (auto* L : graph.sorted) {
        PackedHost p;
        try {
            L->packWeights(p);
        } catch (std::exception& e) {
            err = L->name + ": " + e.what();
            return false;
        }
        if (p.kind) {
            total += p.device_bytes();
            packed.emplace_back(L, std::move(p));
        }
        if (L->typeName == "InstanceNorm") {
            static_cast<InstanceNormLayer*>(L)->computeScratch(N);
            scratchTotal += (L->scratchBytes() + 255) & ~(size_t) 255;
        }
    }
    arenaBytes = total ? total : 256;
    if (cudaMalloc(&arena, arenaBytes) != cudaSuccess) {
        err = "cudaMalloc(weight arena) failed";
        return false;
    }
    {
        char* cur = (char*) arena;
        for (auto& pr : packed) {
            if (place_weights(ctx, pr.second, cur, &pr.first->weights)) {
                err = get_error();
                return false;
            }
            cur += pr.first->weights.bytes;
        }
    }
    if (scratchTotal) {
        if (cudaMalloc(&scratchArena, scratchTotal) != cudaSuccess) {
            err = "cudaMalloc(scratch) failed";
            return false;
        }
        char* cur = (char*) scratchArena;
        for (auto* L : graph.sorted)
            if (L->scratchBytes()) {
                L->scratch = (float*) cur;
                cur += (L->scratchBytes() + 255) & ~(size_t) 255;
            }
    }

    // ---- io staging (stable addresses so the captured graph stays valid) ----
    size_t maxFloats = 1;
    for (auto* L : inputLayers) maxFloats = std::max(maxFloats, L->output->pixels() * (size_t) L->output->c);
    for (auto* L : outputLayers)
        if (L->output) maxFloats = std::max(maxFloats, L->output->pixels() * (size_t) L->output->c);
    ioStageBytes = maxFloats * sizeof(float);
    if (cudaMalloc(&ioStage, ioStageBytes) != cudaSuccess || cudaMalloc(&argmaxDev, sizeof(int) * N) != cudaSuccess) {
        err = "cudaMalloc(io staging) failed";
        return false;
    }
    if (yolo) {
        const size_t yb = yolo->candidateBytes();
        if (cudaMalloc(&yoloDev, yb) != cudaSuccess || cudaMallocHost(&yoloHost, yb) != cudaSuccess) {
            err = "cudaMalloc(YOLO candidate lists) failed";
            return false;
        }
    }
    {
        GenericModelLayer* last = nullptr;
        for (auto* L : outputLayers)
            if (L->output) {
                last = L;
                break;
            }
        isClassifier = last && last->output->h == 1 && last->output->w == 1 && last->output->c > 1;
    }

    // ---- one eager pass: counts launches and warms everything up; then optionally capture ----
    const uint64_t before = ctx->launches;
    if (enqueueForward(false)) {
        err = get_error();
        return false;
    }
    launchesPerForward = (int) (ctx->launches - before);
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
        err = std::string("first forward pass failed: ") + cudaGetErrorString(cudaGetLastError());
        return false;
    }
    if (options.useCudaGraph) {
        const uint64_t keep = ctx->launches;
        if (cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
            err = "cudaStreamBeginCapture failed";
            return false;
        }
        const int rc = enqueueForward(false);
        cudaError_t e = cudaStreamEndCapture(ctx->stream, &cuGraph);
        ctx->launches = keep;
        if (rc || e != cudaSuccess) {
            err = rc ? get_error() : "cudaStreamEndCapture failed";
            return false;
        }
        if (cudaGraphInstantiate(&cuGraphExec, cuGraph, 0) != cudaSuccess) {
            err = "cudaGraphInstantiate failed";
            return false;
        }
    }
    return true;
}

int MixedInferenceCore::enqueueForward(bool) {
    ExecOptions eo;
    eo.convAlgo = options.convAlgo, eo.precision = options.precision;
    // SNNB_SYNC_LAYERS: debugging aid - wait for every layer and name the one whose kernel faulted (eager passes only)
    static const bool syncLayers = getenv("SNNB_SYNC_LAYERS") != nullptr;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (syncLayers) cudaStreamIsCapturing(ctx->stream, &cap);
    const bool capturing = cap != cudaStreamCaptureStatusNone;
    for (auto* L : graph.sorted) {
        if (L->fusedAway || L->isInputLayer || L->typeName == "YOLO") continue;
        if (int rc = L->run(ctx, eo)) return rc;
        if (syncLayers && !capturing) {
            const cudaError_t e = cudaStreamSynchronize(ctx->stream);
            if (e != cudaSuccess) {
                set_error("%s (%s): %s", L->name.c_str(), ctx->last_kernel ? ctx->last_kernel : "?", cudaGetErrorString(e));
                return 1;
            }
        }
    }
    return 0;
}

int MixedInferenceCore::forward() {
    if (cuGraphExec) {
        SNNB_CUDA_OK(cudaGraphLaunch(cuGraphExec, ctx->stream));
        ctx->launches += (uint64_t) launchesPerForward;
        return 0;
    }
    return enqueueForward(false);
}

int MixedInferenceCore::setInput(int idx, const float* host) {
    SNNB_REQUIRE(idx >= 0 && idx < (int) inputLayers.size() && host, "setInput: bad argument");
    snnb_tensor* t     = inputLayers[idx]->output;
    const size_t bytes = t->pixels() * t->c * sizeof(float);
    SNNB_CUDA_OK(cudaMemcpyAsync(ioStage, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return launch_split_f32(ctx, ioStage, t);
}

int MixedInferenceCore::getOutput(int idx, float* host, size_t capacityFloats) {
    SNNB_REQUIRE(idx >= 0 && idx < (int) outputLayers.size() && host, "getOutput: bad argument");
    GenericModelLayer* L = outputLayers[idx];
    if (L->typeName == "YOLO") { // rows of image 0 .. N-1 are fetched with snnb_model_get_boxes
        set_error("getOutput: output %d is a YOLO detection list; use snnb_model_get_boxes", idx);
        return 2;
    }
    snnb_tensor* t      = L->output;
    const size_t floats = t->pixels() * t->c;
    SNNB_REQUIRE(capacityFloats >= floats, "getOutput: buffer too small (%zu < %zu floats)", capacityFloats, floats);
    if (launch_merge_f32(ctx, t, ioStage)) return 1;
    SNNB_CUDA_OK(cudaMemcpyAsync(host, ioStage, floats * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    SNNB_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int MixedInferenceCore::run(const float* hostInput, float* hostOutput, size_t capacityFloats, int* classes1) {
    if (setInput(0, hostInput)) return 1;
    if (forward()) return 1;
    if (yolo && decodeYolo(yoloDev, yoloHost, true)) return 1;
    int outIdx = -1;
    for (size_t i = 0; i < outputLayers.size(); ++i)
        if (outputLayers[i]->typeName != "YOLO") {
            outIdx = (int) i;
            break;
        }
    if (classes1 && isClassifier && outIdx >= 0) {
        if (launch_argmax(ctx, outputLayers[outIdx]->output, argmaxDev)) return 1;
        SNNB_CUDA_OK(cudaMemcpyAsync(classes1, argmaxDev, sizeof(int) * options.batch, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (hostOutput && outIdx >= 0) {
        if (getOutput(outIdx, hostOutput, capacityFloats)) return 1;
    } else {
        SNNB_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    }
    if (classes1 && isClassifier && outIdx >= 0)
        for (uint32_t i = 0; i < options.batch; ++i) classes1[i] += 1; // core.cpp:228-233: argmax + 1
    return 0;
}

// YOLO decode: threshold + compaction on the device (yololayer.cpp:115-164 up to the confidence test), a few KB of candidates
// to the host, then the exact score formula, score sort and NMS there (identical lists, identical order: finishDecode).
int MixedInferenceCore::decodeYolo(void* dev, void* host, bool sync) {
    if (yolo->enqueueCandidates(ctx, dev)) return 1;
    SNNB_CUDA_OK(cudaMemcpyAsync(host, dev, yolo->headBytes(), cudaMemcpyDeviceToHost, ctx->stream)); // count + the first rows
    if (!sync) return 0;
    SNNB_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    const int rc = yolo->finishDecode(host, dev, boxes);
    if (rc < 0) return yolo->decode(ctx, boxes); // an image overflowed its candidate list: all-host decode of the (still resident) heads
    return rc;
}

// ---- streaming (additive to the reference's synchronous run) ---------------------------------------------------------
int MixedInferenceCore::ensureStreaming() {
    if (copyStream) return 0;
    SNNB_CUDA_OK(cudaStreamCreateWithFlags(&copyStream, cudaStreamNonBlocking));
    for (auto& sl : slots) {
        SNNB_CUDA_OK(cudaMalloc(&sl.stageIn, ioStageBytes));
        SNNB_CUDA_OK(cudaMalloc(&sl.stageOut, ioStageBytes));
        SNNB_CUDA_OK(cudaMalloc(&sl.argmax, sizeof(int) * options.batch));
        SNNB_CUDA_OK(cudaHostAlloc(&sl.smallHost, SMALL_RESULT_BYTES, cudaHostAllocMapped));
        SNNB_CUDA_OK(cudaHostGetDevicePointer(&sl.smallDev, sl.smallHost, 0));
        SNNB_CUDA_OK(cudaEventCreateWithFlags(&sl.h2dDone, cudaEventDisableTiming));
        SNNB_CUDA_OK(cudaEventCreateWithFlags(&sl.stageFree, cudaEventDisableTiming));
        SNNB_CUDA_OK(cudaEventCreateWithFlags(&sl.resultReady, cudaEventDisableTiming));
        if (yolo) {
            SNNB_CUDA_OK(cudaMalloc(&sl.yoloDev, yolo->candidateBytes()));
            SNNB_CUDA_OK(cudaMallocHost(&sl.yoloHost, yolo->candidateBytes()));
        }
    }
    return 0;
}

int MixedInferenceCore::submit(const float* hostInput, float* hostOutput, size_t capacityFloats, int* classes1, int* ticket) {
    return submitImpl(hostInput, false, nullptr, nullptr, hostOutput, capacityFloats, classes1, ticket);
}
int MixedInferenceCore::submitU8(const uint8_t* hostInput, const float mean[4], const float norm[4], float* hostOutput, size_t capacityFloats, int* classes1, int* ticket) {
    SNNB_REQUIRE(mean && norm, "submitU8: null mean / norm");
    return submitImpl(hostInput, true, mean, norm, hostOutput, capacityFloats, classes1, ticket);
}
int MixedInferenceCore::submitImage(const snnb_image_io& io, int* ticket) {
    SNNB_REQUIRE(io.input_u8 && io.src_height > 0 && io.src_width > 0, "submit_image: bad input");
    SNNB_REQUIRE(!(io.output_f32 && io.output_u8), "submit_image: choose ONE of output_f32 / output_u8");
    return submitImpl(io.input_u8, true, io.mean4, io.norm4, io.output_f32, io.output_capacity, io.classes_1based, ticket, &io);
}
int MixedInferenceCore::submitImpl(const void* hostInput, bool u8, const float* mean, const float* norm, float* hostOutput, size_t capacityFloats, int* classes1,
                                   int* ticket, const snnb_image_io* io) {
    SNNB_REQUIRE(hostInput && ticket, "submit: null argument");
    if (ensureStreaming()) return 1;
    Slot& sl = slots[nextTicket & 1];
    SNNB_REQUIRE(!sl.busy, "submit: two submissions are already in flight; wait() on ticket %d first", nextTicket - 2);
    int outIdx = 0;
    snnb_tensor* in  = inputLayers[0]->output;
    snnb_tensor* out = outputLayers[outIdx]->output; // nullptr for a detection model: its output is the box list (snnb_model_get_boxes)
    if (!out) hostOutput = nullptr, classes1 = nullptr;
    const bool resize = io && (io->src_height != in->h || io->src_width != in->w);
    const size_t inBytes = resize ? (size_t) in->n * io->src_height * io->src_width * in->c : in->pixels() * in->c * (u8 ? sizeof(uint8_t) : sizeof(float));
    const size_t outFloats = out ? out->pixels() * out->c : 0;
    SNNB_REQUIRE(!hostOutput || capacityFloats >= outFloats, "submit: output buffer too small (%zu < %zu floats)", capacityFloats, outFloats);
    SNNB_REQUIRE(!(io && io->output_u8) || (out && io->output_capacity >= outFloats), "submit_image: u8 output buffer too small or the model has no tensor output");
    void* stage = sl.stageIn;
    if (resize) { // a source image of another size does not fit the model-sized staging: its own buffer, grown on demand
        if (inBytes > sl.stageResizeBytes) {
            SNNB_CUDA_OK(cudaStreamSynchronize(ctx->stream));
            if (sl.stageResize) SNNB_CUDA_OK(cudaFree(sl.stageResize));
            SNNB_CUDA_OK(cudaMalloc(&sl.stageResize, inBytes));
            sl.stageResizeBytes = inBytes;
        }
        stage = sl.stageResize;
    }
    // copy stream: wait until the split kernel of the submission that last used this slot has consumed the staging
    if (sl.everUsed) SNNB_CUDA_OK(cudaStreamWaitEvent(copyStream, sl.stageFree, 0));
    SNNB_CUDA_OK(cudaMemcpyAsync(stage, hostInput, inBytes, cudaMemcpyHostToDevice, copyStream));
    SNNB_CUDA_OK(cudaEventRecord(sl.h2dDone, copyStream));
    // compute stream
    SNNB_CUDA_OK(cudaStreamWaitEvent(ctx->stream, sl.h2dDone, 0));
    if (resize) {
        if (launch_resize_u8(ctx, reinterpret_cast<const uint8_t*>(stage), io->src_height, io->src_width, in, mean, norm, io->linear_filter != 0)) return 1;
    } else if (u8 ? launch_split_u8(ctx, reinterpret_cast<const uint8_t*>(sl.stageIn), in, mean, norm) : launch_split_f32(ctx, sl.stageIn, in)) {
        return 1;
    }
    SNNB_CUDA_OK(cudaEventRecord(sl.stageFree, ctx->stream));
    if (forward()) return 1;
    sl.userOut = nullptr, sl.userClasses = nullptr, sl.userFloats = 0;
    // a small classifier result (values + classes) is written straight into mapped pinned memory by ONE kernel; wait() copies it out
    static const bool noSmall = getenv("SNNB_NO_SMALL_RESULT") != nullptr;
    const bool small = !noSmall && isClassifier && !(io && io->output_u8) && (hostOutput || classes1) &&
                       outFloats * sizeof(float) + options.batch * sizeof(int) <= SMALL_RESULT_BYTES;
    if (small) {
        float* vals = static_cast<float*>(sl.smallDev);
        int* cls    = reinterpret_cast<int*>(static_cast<char*>(sl.smallDev) + outFloats * sizeof(float));
        if (launch_result_small(ctx, out, hostOutput ? vals : nullptr, classes1 ? cls : nullptr)) return 1;
        sl.userOut = hostOutput, sl.userClasses = classes1, sl.userFloats = outFloats;
        hostOutput = nullptr, classes1 = nullptr; // served
    }
    if (hostOutput) {
        if (launch_merge_f32(ctx, out, sl.stageOut)) return 1;
        SNNB_CUDA_OK(cudaMemcpyAsync(hostOutput, sl.stageOut, outFloats * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (io && io->output_u8) { // the output as an 8-bit image: clamp(round(v * scale + offset), 0, 255) on the device, a quarter of the bytes back
        if (launch_merge_u8(ctx, out, reinterpret_cast<uint8_t*>(sl.stageOut), io->out_scale, io->out_offset)) return 1;
        SNNB_CUDA_OK(cudaMemcpyAsync(io->output_u8, sl.stageOut, outFloats, cudaMemcpyDeviceToHost, ctx->stream));
    }
    sl.classesHost = nullptr;
    if (classes1 && isClassifier) {
        if (launch_argmax(ctx, out, sl.argmax)) return 1;
        SNNB_CUDA_OK(cudaMemcpyAsync(classes1, sl.argmax, sizeof(int) * options.batch, cudaMemcpyDeviceToHost, ctx->stream));
        sl.classesHost = classes1;
    }
    if (yolo && decodeYolo(sl.yoloDev, sl.yoloHost, false)) return 1; // candidates -> pinned host, asynchronously; NMS in wait()
    SNNB_CUDA_OK(cudaEventRecord(sl.resultReady, ctx->stream));
    sl.busy = sl.everUsed = true;
    *ticket = nextTicket++;
    return 0;
}

int MixedInferenceCore::wait(int ticket) {
    SNNB_REQUIRE(ticket >= 0 && ticket < nextTicket && ticket >= nextTicket - 2, "wait: ticket %d is not in flight", ticket);
    Slot& sl = slots[ticket & 1];
    SNNB_REQUIRE(sl.busy, "wait: ticket %d was already waited for", ticket);
    SNNB_CUDA_OK(cudaEventSynchronize(sl.resultReady));
    if (sl.userOut) std::memcpy(sl.userOut, sl.smallHost, sl.userFloats * sizeof(float));
    if (sl.userClasses) {
        const int* cls = reinterpret_cast<const int*>(static_cast<const char*>(sl.smallHost) + sl.userFloats * sizeof(float));
        for (uint32_t i = 0; i < options.batch; ++i) sl.userClasses[i] = cls[i] + 1; // core.cpp:228-233: argmax + 1
    }
    sl.userOut = nullptr, sl.userClasses = nullptr;
    if (sl.classesHost)
        for (uint32_t i = 0; i < options.batch; ++i) sl.classesHost[i] += 1; // core.cpp:228-233: argmax + 1
    sl.busy = false;
    if (yolo) {
        const int rc = yolo->finishDecode(sl.yoloHost, sl.yoloDev, boxes);
        SNNB_REQUIRE(rc >= 0, "wait: corrupt detection candidate list");
        return rc;
    }
    return 0;
}

int MixedInferenceCore::layerOutput(int layerId, float* host, size_t capacityFloats) {
    SNNB_REQUIRE(layerId >= 0 && layerId < (int) layers.size() && host, "layerOutput: bad argument");
    GenericModelLayer* L = layers[layerId].get();
    SNNB_REQUIRE(!(L->typeName == "Conv2D" && static_cast<Conv2DLayer*>(L)->foldedInto),
                 "layerOutput: layer %d (%s) was fused into the K loop of the convolution it is added to; load the model with fuse=0 to observe it", layerId,
                 L->name.c_str());
    SNNB_REQUIRE(L->output, "layerOutput: layer %d (%s) has no device tensor", layerId, L->name.c_str());
    SNNB_REQUIRE(!(L->typeName == "Conv2D" && static_cast<Conv2DLayer*>(L)->fusedAct >= 0),
                 "layerOutput: layer %d (%s) was fused into its Add; load the model with fuse=0 to observe it", layerId, L->name.c_str());
    SNNB_REQUIRE(!(L->fusedAway && L->typeName == "AveragePooling2D"),
                 "layerOutput: layer %d (%s) was fused into the classifier head (pool + Dense in one launch); load the model with fuse=0 to observe it", layerId,
                 L->name.c_str());
    const size_t floats = L->output->pixels() * L->output->c;
    SNNB_REQUIRE(capacityFloats >= floats, "layerOutput: buffer too small (%zu < %zu floats)", capacityFloats, floats);
    return snnb_tensor_download_nhwc(ctx, L->output, host);
}

int MixedInferenceCore::timeLayers(std::vector<float>& ms) {
    ms.assign(layers.size(), 0.0f);
    std::vector<cudaEvent_t> ev(graph.sorted.size() + 1);
    for (auto& e : ev) SNNB_CUDA_OK(cudaEventCreate(&e));
    ExecOptions eo;
    eo.convAlgo = options.convAlgo, eo.precision = options.precision;
    SNNB_CUDA_OK(cudaEventRecord(ev[0], ctx->stream));
    layerKernels.assign(layers.size(), std::string());
    for (size_t i = 0; i < graph.sorted.size(); ++i) {
        GenericModelLayer* L = graph.sorted[i];
        if (!(L->fusedAway || L->isInputLayer || L->typeName == "YOLO")) {
            ctx->last_kernel = nullptr;
            if (int rc = L->run(ctx, eo)) return rc;
            layerKernels[L->layerId] = ctx->last_kernel ? ctx->last_kernel : (L->typeName + " kernels");
        }
        SNNB_CUDA_OK(cudaEventRecord(ev[i + 1], ctx->stream));
    }
    SNNB_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < graph.sorted.size(); ++i) {
        float t = 0;
        SNNB_CUDA_OK(cudaEventElapsedTime(&t, ev[i], ev[i + 1]));
        ms[graph.sorted[i]->layerId] = t;
    }
    for (auto& e : ev) cudaEventDestroy(e);
    return 0;
}

int MixedInferenceCore::dumpOutputs(const std::string& dir) {
    for (auto& l : layers) {
        if (!l->output || l->fusedAway) continue;
        // a Conv2D fused into its Add writes the ADD's tensor (post-add, post-activation): under the conv's name the file would
        // not be what a reference run dumps for that layer (layerOutput() refuses the same case)
        SNNB_REQUIRE(!(l->typeName == "Conv2D" && l->fusedAct >= 0), "dumpOutputs: %s was fused into its Add; load the model with fuse=0 to dump every layer", l->name.c_str());
        std::string path = dir + "/" + l->name + " pass[0].dump"; // vulkanBackend.cpp:108-143 naming
        if (snnb_tensor_dump(ctx, l->output, path.c_str())) return 1;
    }
    return 0;
}

} // namespace snn
