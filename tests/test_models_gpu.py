"""GPU parity tests, model level: the C++ engine (JSON -> graph -> CUDA) vs the oracle walking the same JSON.

Mirrors the reference's model tests (demo/test/unittest/resnet18Test.cpp:85-198, mobilenetv2Test.cpp:82-211): dump
every layer's output and compare it, layer by layer, with the CPU ground truth — here the oracle instead of ncnn,
tolerance 1e-3 of each tensor's range (assert_layer_close) instead of the reference's 0.01; classification top-1 index
bit-exact. The BASELINE.json configurations are checked AT THEIR SIZE (every layer of a sample of the batch, fused and
unfused, soft-max outputs and pre-soft-max logits) as well as through size-independent properties (batch consistency,
fused == unfused, CUDA-graph replay == eager).
"""
import os

import numpy as np
import pytest

from oracle import oracle
from shadernn_b200 import core, modelzoo

pytestmark = pytest.mark.gpu

EPS = 1e-3


def assert_same_boxes(got, ref, tol=3e-3):
    """Detection lists agree as SETS: equal scores may sort differently (NMS orders by score, yololayer.cpp:73-78)."""
    assert got.shape == ref.shape, (got.shape, ref.shape)
    used = set()
    for r in ref:
        d = np.max(np.abs(got - r) / (np.abs(r) + 1.0), axis=1)
        for j in np.argsort(d):
            if int(j) not in used:
                assert d[j] < tol, (r, got[j], d[j])
                used.add(int(j))
                break


def assert_layer_close(got, want, eps, what):
    """THE parity criterion (north_star: "within 1e-3 relative fp32 per layer"): the largest absolute difference of a layer's
    output is at most eps times the largest magnitude of the reference output, i.e. error relative to the tensor's range.
    Nothing else passes a layer (round 1 also accepted "no element outside the reference's abs-or-rel comparator")."""
    assert got.shape == want.shape, (what, got.shape, want.shape)
    scale = float(np.abs(want).max())
    err = float(np.abs(got.astype(np.float64) - want.astype(np.float64)).max())
    assert err <= eps * max(scale, 1e-30), "%s: max |err| %.3g = %.3g of the tensor's range %.3g (limit %g)" % (what, err, err / max(scale, 1e-30), scale, eps)
    return err / max(scale, 1e-30)


def baseline_size_check(ctx, name, hw, batch, sample, model_dir, fuse, eps=EPS, min_layers=0, precision="fp32x3", **build_kw):
    """Per-layer parity AT BASELINE.json's size (demo/test/unittest/resnet18Test.cpp:85-198 compares its 20 checkpoints at the
    real input size): the engine runs the full batch, the oracle the first `sample` images of the same batch; every layer
    output the engine can show (all of them with fuse=0; with fuse=1 the tensors that survive fusion) must agree."""
    from shadernn_b200._lib import SnnbError
    path, layers = modelzoo.build(name, model_dir, input_hw=hw, **build_kw)
    x = modelzoo.synthetic_input(name, batch, hw)
    want = oracle.Model(path).run(x[:sample], return_all=True)
    m = core.MixedInferenceCore(ctx, path, batch=batch, input_hw=hw, fuse=fuse, use_cuda_graph=fuse, precision=precision)
    m.set_input(x)
    m.forward()
    ctx.sync()
    worst, compared = 0.0, 0
    for i in range(m.num_layers):
        lname, ltype, shape = m.layer_info(i)
        if ltype == "YOLO":
            continue
        try:
            got = m.layer_output(i)
        except SnnbError:
            assert fuse, lname  # only fusion may hide a layer
            continue
        if fuse and layers[i]["type"] in ("ZeroPadding2D", "Flatten"):
            continue  # fused away: an alias of the producer's tensor (a folded Pad, the Flatten of a 1x1 map)
        worst = max(worst, assert_layer_close(got[:sample], want[i], eps, lname))
        compared += 1
    assert compared >= min_layers, (compared, min_layers)
    print("%s %dx%d batch %d fuse=%d %s: %d layers compared, worst max|err|/range %.3g" % (name, hw[0], hw[1], batch, int(fuse), precision, compared, worst))
    return m, x, want, worst


def layerwise_check(ctx, name, hw, batch, model_dir, eps=EPS, **build_kw):
    path, layers = modelzoo.build(name, model_dir, input_hw=hw, **build_kw)
    x = modelzoo.synthetic_input(name, batch, hw)
    om = oracle.Model(path)
    want = om.run(x, return_all=True)
    m = core.MixedInferenceCore(ctx, path, batch=batch, input_hw=hw, fuse=False)
    assert m.num_layers == len(layers)
    m.set_input(x)
    m.forward()
    ctx.sync()
    worst = 0.0
    for i in range(m.num_layers):
        lname, ltype, shape = m.layer_info(i)
        assert ("layer [%02d]" % i) in lname  # dp.cpp:135 naming
        if ltype == "YOLO":
            continue
        assert shape == want[i].shape, (lname, shape, want[i].shape)
        got = m.layer_output(i)
        worst = max(worst, assert_layer_close(got, want[i], eps, lname))
    return m, om, x, want, worst


def test_espcn_layerwise_and_embedded_weights(ctx, model_dir):
    # BASELINE configs[0]: ESPCN 2x, 224x224x1, batch 1 (embedded-JSON weights path of the parser)
    m, om, x, want, worst = layerwise_check(ctx, "espcn", (224, 224), 1, model_dir)
    out, _ = m.run(x, want_classes=False)
    assert out.shape == (1, 448, 448, 1)
    assert oracle.compare(out, want[-1], EPS) == 0
    assert worst < 1e-4


def test_resnet18_layerwise_and_top1(ctx, model_dir):
    m, om, x, want, worst = layerwise_check(ctx, "resnet18", (64, 64), 4, model_dir)
    out, cls = m.run(x)
    assert out.shape == (4, 1, 1, 10)
    assert np.array_equal(cls, oracle.argmax1(want[-1]))  # 1-based class index, bit-exact (core.cpp:228-233)
    assert np.allclose(out.sum(axis=-1), 1.0, atol=1e-4)  # softmax rows


# The product forms of the tensor-core path (snnb.h). "fp32x3" = fp16 hi+lo pairs for activations AND weights: fp32-class, THE
# parity mode, held to 3e-4 (measured <= 2.0e-4) against the 1e-3 bar. "fp16w" = weights rounded once to fp16 (2 MMAs per product):
# an opt-in fast mode that does NOT meet the bar everywhere - convolution layers measure 2e-4 .. 7e-4 of their range but the
# error accumulates with depth: 4.0e-3 at ResNet-18's soft-max output, 6.5e-3 inside MobileNetV2 (72 layers) - so it is only held
# to 2e-2 here (a guard against gross errors) and is never the headline (DESIGN.md section 3.6 has the measured rejection).
LIMIT = {"fp32x3": 3e-4, "fp16w": 2e-2}


@pytest.mark.parametrize("fuse,precision", [(False, "fp32x3"), (True, "fp32x3"), (False, "fp16w"), (True, "fp16w")])
def test_resnet18_baseline_size_every_layer(ctx, model_dir, fuse, precision):
    # BASELINE.json configs[1]: ResNet-18 224x224x3, batch 32. Every layer of a 4-image sample vs the oracle, fuse=0 and fuse=1
    m, x, want, worst = baseline_size_check(ctx, "resnet18", (224, 224), 32, 4, model_dir, fuse, min_layers=20 if fuse else 33, precision=precision, eps=LIMIT[precision])
    out, cls = m.run(x)
    assert np.array_equal(cls[:4], oracle.argmax1(want[-1]))
    assert len(set(cls.tolist())) >= 5, cls  # the arg-max is decided by the image (round 1: one constant class)
    assert float(out.max()) < 0.999  # ... and the soft-max is not saturated
    assert worst < LIMIT[precision]


@pytest.mark.parametrize("precision", ["fp32x3", "fp16w"])
def test_resnet18_baseline_size_logits(ctx, model_dir, precision):
    # the pre-soft-max logits of the same graph, all 32 images (the oracle needs ~1.5 s per 8 images on 8 cores)
    path, _ = modelzoo.build("resnet18", model_dir + "/lin", input_hw=(224, 224), head_activation="linear")
    x = modelzoo.synthetic_input("resnet18", 32, (224, 224))
    want = oracle.Model(path).run(x).reshape(32, 10)
    m = core.MixedInferenceCore(ctx, path, batch=32, fuse=True, use_cuda_graph=True, precision=precision)
    out, cls = m.run(x)
    rel = assert_layer_close(out.reshape(32, 10), want, LIMIT[precision], "ResNet-18 logits")
    print("ResNet-18 224x224 batch 32 logits, %s: max|err|/range %.3g" % (precision, rel))
    assert rel < LIMIT[precision]
    assert np.array_equal(cls - 1, want.argmax(1))
    assert len(set(want.argmax(1).tolist())) >= 5


@pytest.mark.parametrize("fuse,precision", [(False, "fp32x3"), (True, "fp32x3"), (True, "fp16w")])
def test_mobilenetv2_baseline_size_every_layer(ctx, model_dir, fuse, precision):
    # BASELINE.json configs[2]: MobileNetV2 224x224x3, batch 64 (1000 classes); 2-image sample
    m, x, want, worst = baseline_size_check(ctx, "mobilenetv2", (224, 224), 64, 2, model_dir, fuse, min_layers=50 if fuse else 72, precision=precision, eps=LIMIT[precision])
    out, cls = m.run(x)
    assert np.array_equal(cls[:2], oracle.argmax1(want[-1]))
    assert len(set(cls.tolist())) >= 8, cls
    assert worst < LIMIT[precision]


@pytest.mark.parametrize("precision", ["fp32x3", "fp16w"])
def test_yolov3tiny_baseline_size_every_layer(ctx, model_dir, precision):
    # BASELINE.json configs[3]: YOLOv3-tiny 416x416x3, batch 16; 1-image sample
    m, x, want, worst = baseline_size_check(ctx, "yolov3tiny", (416, 416), 16, 1, model_dir, False, min_layers=20, precision=precision, eps=LIMIT[precision])
    assert worst < LIMIT[precision]


@pytest.mark.parametrize("fuse,precision", [(False, "fp32x3"), (True, "fp32x3"), (True, "fp16w")])
def test_candy_baseline_size_every_layer(ctx, model_dir, fuse, precision):
    # BASELINE.json configs[4]'s per-GPU shard: Candy 720x720x3, one image (inputs in [0,255])
    m, x, want, worst = baseline_size_check(ctx, "candy", (720, 720), 1, 1, model_dir, fuse, min_layers=35, precision=precision, eps=LIMIT[precision])
    assert worst < LIMIT[precision]


def test_mobilenetv2_layerwise(ctx, model_dir):
    m, om, x, want, worst = layerwise_check(ctx, "mobilenetv2", (96, 96), 2, model_dir, classes=100)
    out, cls = m.run(x)
    assert np.array_equal(cls, oracle.argmax1(want[-1]))


def test_yolov3tiny_layerwise_and_boxes(ctx, model_dir):
    m, om, x, want, worst = layerwise_check(ctx, "yolov3tiny", (416, 416), 1, model_dir)
    m.run(x, want_classes=False)
    assert_same_boxes(m.boxes(0), om.boxes[0])


def test_yolo_decode_with_planted_detection(ctx, model_dir):
    # random heads rarely cross the 0.35 threshold; plant a confident cell through the final conv bias instead
    path, layers = modelzoo.build("yolov3tiny", model_dir, input_hw=(416, 416), seed=11)
    head = [l for l in layers if l["type"] == "Conv2D" and l["outputPlanes"] == 18][0]
    head["_w"]["bias"][:] = 0
    head["_w"]["bias"][4] = 6.0  # objectness
    head["_w"]["bias"][5] = 6.0  # class logit
    modelzoo.write_model(layers, path, split=True)
    x = modelzoo.synthetic_input("yolov3tiny", 1, (416, 416))
    om = oracle.Model(path)
    om.run(x)
    m = core.MixedInferenceCore(ctx, path, batch=1)
    m.run(x, want_classes=False)
    got, ref = m.boxes(0), om.boxes[0]
    assert len(ref) > 0
    assert_same_boxes(got, ref)


def test_yolo_device_compaction_streaming_and_batch(ctx, model_dir):
    # decode = threshold + compaction on the device, exact formula + NMS on the host (yololayer.cpp:56-164): the lists must be
    # those of the oracle (which decodes everything on the CPU), image by image, through run() AND through submit()/wait()
    import ctypes as C
    path, layers = modelzoo.build("yolov3tiny", model_dir + "/planted", input_hw=(416, 416), seed=21)
    for head in [l for l in layers if l["type"] == "Conv2D" and l["outputPlanes"] == 18]:
        head["_w"]["bias"][:] = 0
        head["_w"]["bias"][[4, 5, 10, 11]] = [-1.0, 0.0, -1.0, 0.0]  # scores scattered around the 0.35 threshold
    modelzoo.write_model(layers, path, split=True)
    xs = [modelzoo.synthetic_input("yolov3tiny", 4, (416, 416), seed=s) for s in (1, 2, 3)]
    om = oracle.Model(path)
    m = core.MixedInferenceCore(ctx, path, batch=4, fuse=True, use_cuda_graph=True)
    refs = []
    for x in xs:
        om.run(x)
        refs.append([b.copy() for b in om.boxes])
        m.run(x, want_classes=False)
        for n in range(4):
            assert_same_boxes(m.boxes(n), refs[-1][n])
    assert sum(len(b) for r in refs for b in r) > 20, "the planted heads should produce detections"
    assert any(len(b) != len(refs[0][0]) for r in refs for b in r), "images should differ in their detection count"
    ins = [np.ascontiguousarray(x) for x in xs]
    pending = None
    for i, x in enumerate(ins):
        t = m.submit_raw(x.ctypes.data_as(C.c_void_p), None, 0, None)
        if pending is not None:
            m.wait(pending[0])  # boxes of the PREVIOUS submission
            for n in range(4):
                assert_same_boxes(m.boxes(n), refs[pending[1]][n])
        pending = (t, i)
    m.wait(pending[0])
    for n in range(4):
        assert_same_boxes(m.boxes(n), refs[pending[1]][n])


def test_candy_layerwise(ctx, model_dir):
    # reflect padding, instance norm, nearest upsample, residual adds; inputs in [0,255]
    layerwise_check(ctx, "candy", (64, 64), 1, model_dir)


@pytest.mark.parametrize("name,hw,kw", [("resnet18", (96, 96), {}), ("mobilenetv2", (96, 96), {"classes": 50}), ("candy", (48, 48), {})])
def test_fused_graph_equals_unfused_and_graph_replay(ctx, model_dir, name, hw, kw):
    path, _ = modelzoo.build(name, model_dir, input_hw=hw, **kw)
    x = modelzoo.synthetic_input(name, 3, hw)
    plain = core.MixedInferenceCore(ctx, path, batch=3, input_hw=hw, fuse=False)
    fused = core.MixedInferenceCore(ctx, path, batch=3, input_hw=hw, fuse=True)
    graph = core.MixedInferenceCore(ctx, path, batch=3, input_hw=hw, fuse=True, use_cuda_graph=True)
    o0, c0 = plain.run(x, want_classes=name != "candy")
    o1, c1 = fused.run(x, want_classes=name != "candy")
    o2, c2 = graph.run(x, want_classes=name != "candy")
    o3, _ = graph.run(x, want_classes=False)  # replay twice: idempotent
    assert fused.launches_per_forward <= plain.launches_per_forward
    if name != "candy":  # candy has no Conv->Add chains or standalone pads to fuse (adds follow InstanceNorm)
        assert fused.launches_per_forward < plain.launches_per_forward
    scale = max(1.0, float(np.abs(o0).max()))
    # same arithmetic, but a fused conv+add skips one split-bf16 rounding (2^-17) of the intermediate per block
    assert float(np.abs(o1 - o0).max()) / scale < 1e-4
    assert np.array_equal(o2, o1) and np.array_equal(o3, o2)
    if c0 is not None:
        assert np.array_equal(c0, c1) and np.array_equal(c1, c2)


# ---- half-precision storage mode (SURVEY §8 f-N4): the reference's preferrHalfPrecision / RGBA16F textures ------------------
HALF_TOL = 0.1  # the reference's own half-precision threshold (demo/common/testutil.h:1195), relative to each tensor's range


@pytest.mark.parametrize("name,hw,batch,sample", [("resnet18", (224, 224), 32, 2), ("mobilenetv2", (224, 224), 16, 2), ("yolov3tiny", (416, 416), 2, 1),
                                                  ("candy", (256, 256), 1, 1), ("espcn", (224, 224), 1, 1)])
def test_fp16_storage_mode_every_layer(ctx, model_dir, name, hw, batch, sample):
    # one fp16 plane per tensor and per weight, one MMA per product, half the bytes: every layer within the reference's
    # half-precision tolerance, and for the classifiers the same top-1 as the fp32-class oracle
    m, x, want, worst = baseline_size_check(ctx, name, hw, batch, sample, model_dir, True, eps=HALF_TOL, precision="fp16")
    if name in ("resnet18", "mobilenetv2"):
        out, cls = m.run(x)
        assert np.array_equal(cls[:sample], oracle.argmax1(want[-1]))
    assert worst < 0.02, worst  # measured: ~1e-3 .. 1e-2, an order of magnitude inside the reference's 0.1


def _real_candy_head(tmp_dir):
    from _candy_fixture import head_graph as _head_graph
    from shadernn_b200 import onnx2snn
    g, x, want = _head_graph()
    layers = onnx2snn.convert_graph(g, input_hw=(64, 64))
    return modelzoo.write_model(layers, os.path.join(tmp_dir, "candy_head_layers.json"), split=True), x, want


@pytest.mark.parametrize("precision", ["fp32x3", "fp16w"])
def test_real_candy_weights_head_vs_torch_golden(ctx, tmp_path, precision):
    # REFERENCE-HELD WEIGHTS (the first two stages of modelzoo/StyleTransfer/candy-9_simplified.onnx, frozen in
    # tests/golden/candy_head_golden.npz) against what torch computed for those ONNX nodes: 9x9 and 3x3-stride-2 convolutions
    # with reflect padding, InstanceNorm, ReLU - on the CUDA engine, through the converter's JSON
    path, x, want = _real_candy_head(str(tmp_path))
    m = core.MixedInferenceCore(ctx, path, batch=1, input_hw=(64, 64), fuse=True, precision=precision)
    out, _ = m.run(x, want_classes=False)
    rel = assert_layer_close(out, want, LIMIT[precision], "real Candy head")
    print("real Candy weights, first two stages, %s: max|err|/range %.3g" % (precision, rel))
    assert rel < LIMIT[precision]


@pytest.fixture(scope="module")
def candy_whole(tmp_path_factory):
    # the reference's whole candy-9_simplified.onnx as tests/_candy_fixture.py writes it (its graph, its 1-D initialisers,
    # seeded convolution kernels), converted at 224x224, and torch's evaluation of that ONNX graph
    from _candy_fixture import whole_model_onnx
    from shadernn_b200 import onnx2snn
    d = tmp_path_factory.mktemp("candy_whole")
    src = whole_model_onnx(str(d / "candy-9_simplified.onnx"))
    path, _ = onnx2snn.convert(src, str(d), input_hw=(224, 224))
    x = modelzoo.synthetic_input("candy", 1, (224, 224))
    return path, x, onnx2snn.torch_eval(onnx2snn.load_onnx(src), x)


@pytest.mark.parametrize("precision", ["fp32x3", "fp16w"])
def test_real_candy_whole_model_vs_torch_and_oracle(ctx, candy_whole, precision):
    # the WHOLE model converted from the reference's ONNX file: final image against torch's evaluation of the ONNX graph and
    # every layer against the oracle
    path, x, want = candy_whole
    layers_want = oracle.Model(path).run(x, return_all=True)
    m = core.MixedInferenceCore(ctx, path, batch=1, fuse=False, precision=precision)
    m.set_input(x)
    m.forward()
    ctx.sync()
    worst = 0.0
    for i in range(m.num_layers):
        worst = max(worst, assert_layer_close(m.layer_output(i), layers_want[i], LIMIT[precision], m.layer_info(i)[0]))
    out, _ = m.run(x, want_classes=False)
    rel = assert_layer_close(out, want, LIMIT[precision], "real Candy output vs torch(ONNX)")
    print("real Candy 224x224, %s: per-layer worst vs oracle %.3g, output vs torch(ONNX) %.3g" % (precision, worst, rel))
    assert max(worst, rel) < LIMIT[precision]


def test_batch_consistency_at_baseline_size(ctx, model_dir):
    # size-independent property at BASELINE.json's full ResNet-18 config (224x224x3, batch 32): every image's logits
    # equal what the same image yields in a batch of 1. No kernel reduces across images; the only difference allowed is
    # fp32 association in layers whose K loop is split differently at the two batch sizes (split-K on the 7x7 maps),
    # orders of magnitude below the 1e-3 parity bar. The class index must be identical.
    path, _ = modelzoo.build("resnet18", model_dir, input_hw=(224, 224))
    x = modelzoo.synthetic_input("resnet18", 32, (224, 224))
    big = core.MixedInferenceCore(ctx, path, batch=32, fuse=True, use_cuda_graph=True)
    out, cls = big.run(x)
    one = core.MixedInferenceCore(ctx, path, batch=1, fuse=True)
    for i in (0, 13, 31):
        o1, c1 = one.run(x[i:i + 1])
        assert c1[0] == cls[i]
        assert float(np.abs(o1[0] - out[i]).max()) <= 2e-5 * max(1.0, float(np.abs(out[i]).max()))
    assert np.all((cls >= 1) & (cls <= 10))


def test_u8_input_normalised_on_device(ctx, model_dir):
    # snnb_model_submit_u8 = ImageTexture::convertToRGBA32FAndNormalize on the device (imageTexture.h:114) + the fp32 path:
    # identical logits to feeding (u8 - mean) * norm as fp32 (ResNet-18 constants of demo/common/modelInference.cpp:135)
    path, _ = modelzoo.build("resnet18", model_dir, input_hw=(64, 64))
    m = core.MixedInferenceCore(ctx, path, batch=3, input_hw=(64, 64), fuse=True, use_cuda_graph=True)
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (3, 64, 64, 3), dtype=np.uint8)
    mean, norm = [127.5] * 4, [1.0 / 127.5] * 4
    ref, cref = m.run((img.astype(np.float32) - np.float32(127.5)) * np.float32(1.0 / 127.5))
    out, cls = m.run_u8(img, mean, norm)
    assert np.array_equal(cls, cref)
    assert float(np.abs(out - ref).max()) <= 1e-6 * max(1.0, float(np.abs(ref).max()))
    # per-channel constants (index c & 3)
    mean2, norm2 = [10.0, 20.0, 30.0, 0.0], [0.01, 0.02, 0.03, 1.0]
    ref2, _ = m.run((img.astype(np.float32) - np.array(mean2[:3], np.float32)) * np.array(norm2[:3], np.float32))
    out2, _ = m.run_u8(img, mean2, norm2)
    assert float(np.abs(out2 - ref2).max()) <= 1e-5 * max(1.0, float(np.abs(ref2).max()))


def test_model_error_paths(ctx, tmp_path):
    from shadernn_b200._lib import SnnbError
    with pytest.raises(SnnbError):
        core.MixedInferenceCore(ctx, str(tmp_path / "missing.json"))
    bad = tmp_path / "bad.json"
    bad.write_text('{"numLayers": {"count": 1}, "Layer_0": {"type": "NoSuchLayer", "numInputs": 0, "inputId": [], "outputPlanes": 3}}')
    with pytest.raises(SnnbError) as e:
        core.MixedInferenceCore(ctx, str(bad))
    assert "Not found layer" in str(e.value)  # layerFactory.cpp:155-157
    # declared planes that disagree with the graph are load errors, not device faults (ADVICE r1)
    import json
    path, _ = modelzoo.build("espcn", str(tmp_path), input_hw=(32, 32))
    root = json.load(open(path))
    root["Layer_2"]["inputPlanes"] = 8  # the producer has 16 channels; weights shrunk to match the declaration
    root["Layer_2"]["weights"]["kernel"] = root["Layer_2"]["weights"]["kernel"][:16 * 8 * 9]
    lie = tmp_path / "lie.json"
    lie.write_text(json.dumps(root))
    with pytest.raises(SnnbError) as e:
        core.MixedInferenceCore(ctx, str(lie), input_hw=(32, 32))
    assert "inputPlanes" in str(e.value)
    trunc = tmp_path / "trunc.json"
    trunc.write_text('{"numLayers": {"count": 2}')
    with pytest.raises(SnnbError):
        core.MixedInferenceCore(ctx, str(trunc))


@pytest.mark.parametrize("linear", [True, False])
def test_device_resize_normalise_and_u8_output(ctx, model_dir, linear):
    # SURVEY §8 f-N3: pre/post-processing on the device. snnb_model_submit_image takes 8-bit images of any size, resizes them like
    # ImageTexture::resize (vk_resize.comp:42-61), normalises, runs the model and can return an 8-bit image
    # (clamp(round(v * scale + offset))). Checked against the oracle's restatement of the resize + the same model fed with the
    # resized fp32 image through the plain run().
    path, _ = modelzoo.build("candy", model_dir, input_hw=(64, 80))
    m = core.MixedInferenceCore(ctx, path, batch=2, input_hw=(64, 80), fuse=True)
    rng = np.random.default_rng(9)
    img = rng.integers(0, 256, (2, 150, 233, 3), dtype=np.uint8)
    mean4, norm4 = [10.0, 20.0, 30.0, 0.0], [1.0, 0.5, 2.0, 1.0]
    resized = oracle.resize_normalize(img, (64, 80), mean4, norm4, linear)
    want, _ = m.run(resized, want_classes=False)
    got, _ = m.run_image(img, mean4, norm4, linear=linear)
    assert got.shape == want.shape
    assert float(np.abs(got - want).max()) <= 2e-4 * float(np.abs(want).max())  # resize arithmetic agrees to fp32 rounding
    # the resized input itself, observed through an identity-sized run: up-scaling too
    up = oracle.resize_normalize(img[:, :40, :50], (64, 80), [0.0] * 4, [1.0] * 4, linear)
    got_up, _ = m.run_image(img[:, :40, :50].copy(), [0.0] * 4, [1.0] * 4, linear=linear)
    want_up, _ = m.run(up, want_classes=False)
    assert float(np.abs(got_up - want_up).max()) <= 2e-4 * float(np.abs(want_up).max())
    # 8-bit output
    scale, offset = 0.7, 12.0
    got_u8, _ = m.run_image(img, mean4, norm4, linear=linear, out_u8=True, out_scale=scale, out_offset=offset)
    want_u8 = np.clip(np.rint(got * np.float32(scale) + np.float32(offset)), 0, 255).astype(np.uint8)
    assert got_u8.dtype == np.uint8 and int(np.abs(got_u8.astype(int) - want_u8.astype(int)).max()) <= 1
    assert float((got_u8 != want_u8).mean()) < 1e-3  # only exact .5 ties may round differently


def test_layer_registration_through_the_c_abi(ctx, tmp_path):
    # snnb_register_layer = snn::dp::registerLayer(name, LayerCreator) (layerFactory.h:116-122) at the C boundary: the host registers
    # a creator for a new layer type; the model file names it; the creator reads its JSON through the accessors and supplies dims +
    # launches. Here: "GatedSiLU" = SiLU of the input through the library's own activation launch, output dims = input dims.
    import ctypes as C
    import json

    from shadernn_b200._lib import SnnbError, lib
    DIMS = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int))
    RUN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_void_p)
    DESTROY = C.CFUNCTYPE(None, C.c_void_p)

    class Impl(C.Structure):
        _fields_ = [("user", C.c_void_p), ("output_dims", DIMS), ("run", RUN), ("destroy", DESTROY)]

    CREATOR = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.POINTER(Impl))
    seen = {}

    def dims(user, n, in_hwc, out_hwc):
        for k in range(3):
            out_hwc[k] = in_hwc[k]
        return 0

    def run(user, ctx_h, n, inputs, output):
        seen["runs"] = seen.get("runs", 0) + 1
        return lib().snnb_activation_launch(ctx_h, core.ACT["SiLU"], 0.0, inputs[0], output)

    keep = [DIMS(dims), RUN(run), DESTROY(lambda u: seen.__setitem__("destroyed", seen.get("destroyed", 0) + 1))]

    def creator(reg_user, layer, out):
        num, buf = C.c_double(), C.create_string_buffer(32)
        data, cnt = C.POINTER(C.c_double)(), C.c_size_t()
        assert lib().snnb_layer_json_number(layer, b"gain", C.byref(num)) == 0 and num.value == 2.5
        assert lib().snnb_layer_json_string(layer, b"flavour", buf, 32) == 0 and buf.value == b"sweet"
        assert lib().snnb_layer_json_numbers(layer, b"weights.table", C.byref(data), C.byref(cnt)) == 0 and [data[i] for i in range(cnt.value)] == [1.0, 2.0, 3.0]
        assert lib().snnb_layer_json_number(layer, b"missing", C.byref(num)) != 0
        out[0].user, out[0].output_dims, out[0].run, out[0].destroy = None, keep[0], keep[1], keep[2]
        seen["created"] = seen.get("created", 0) + 1
        return 0

    cb = CREATOR(creator)
    model = {"numLayers": {"count": 2},
             "Layer_0": {"type": "InputLayer", "name": "input_1", "Input Width": 12, "Input Height": 10, "outputPlanes": 5, "inputPlanes": 5, "numInputs": 0, "inputId": [],
                         "inputIndex": 0},
             "Layer_1": {"type": "GatedSiLU", "name": "gated", "inputPlanes": 5, "outputPlanes": 5, "numInputs": 1, "inputId": [0], "gain": 2.5, "flavour": "sweet",
                         "weights": {"table": [1, 2, 3]}}}
    path = tmp_path / "custom.json"
    path.write_text(json.dumps(model))
    with pytest.raises(SnnbError) as e:  # unknown until registered (layerFactory.cpp:155-157)
        core.MixedInferenceCore(ctx, str(path), batch=2)
    assert "Not found layer" in str(e.value)
    assert lib().snnb_register_layer(b"GatedSiLU", C.cast(cb, C.c_void_p), None) == 0
    try:
        m = core.MixedInferenceCore(ctx, str(path), batch=2)
        x = np.random.default_rng(3).uniform(-3, 3, (2, 10, 12, 5)).astype(np.float32)
        out, _ = m.run(x, want_classes=False)
        want = x / (1.0 + np.exp(-x))
        assert out.shape == x.shape and float(np.abs(out - want).max()) < 1e-5
        assert seen["created"] == 1 and seen["runs"] >= 2  # init's eager pass + the run
        m.close()
        assert seen.get("destroyed") == 1
    finally:
        assert lib().snnb_unregister_layer(b"GatedSiLU") == 0
    assert lib().snnb_unregister_layer(b"GatedSiLU") != 0


def test_streaming_submit_wait_matches_synchronous_run(ctx, model_dir):
    # snnb_model_submit / snnb_model_wait: double-buffered pipeline, results identical to run(), tickets enforce depth 2
    import ctypes as C

    from shadernn_b200._lib import SnnbError
    path, _ = modelzoo.build("resnet18", model_dir, input_hw=(64, 64))
    m = core.MixedInferenceCore(ctx, path, batch=4, input_hw=(64, 64), fuse=True, use_cuda_graph=True)
    xs = [modelzoo.synthetic_input("resnet18", 4, (64, 64), seed=s) for s in range(5)]
    want = [m.run(x) for x in xs]
    outs = [np.empty(m.output_shape(0), np.float32) for _ in xs]
    clss = [(C.c_int * 4)() for _ in xs]
    ins = [np.ascontiguousarray(x) for x in xs]
    tickets = []
    for i in range(5):
        t = m.submit_raw(ins[i].ctypes.data_as(C.c_void_p), outs[i].ctypes.data_as(C.c_void_p), outs[i].size, clss[i])
        tickets.append(t)
        if i >= 1:
            m.wait(tickets[i - 1])
    with pytest.raises(SnnbError):
        m.wait(tickets[0])  # already consumed
    m.wait(tickets[-1])
    for i in range(5):
        assert np.array_equal(outs[i], want[i][0])
        assert list(clss[i]) == list(want[i][1])
    # a third submission without waiting is refused
    t0 = m.submit_raw(ins[0].ctypes.data_as(C.c_void_p), outs[0].ctypes.data_as(C.c_void_p), outs[0].size, clss[0])
    t1 = m.submit_raw(ins[1].ctypes.data_as(C.c_void_p), outs[1].ctypes.data_as(C.c_void_p), outs[1].size, clss[1])
    with pytest.raises(SnnbError):
        m.submit_raw(ins[2].ctypes.data_as(C.c_void_p), outs[2].ctypes.data_as(C.c_void_p), outs[2].size, clss[2])
    m.wait(t0)
    m.wait(t1)


@pytest.mark.parametrize("name", ["resnet18", "mobilenet_v2"])
def test_torchvision_export_runs_like_torch(ctx, tmp_path, name):
    # independent cross-check (SURVEY §8c "torch-CPU as a secondary check"): a torchvision module exported with
    # shadernn_b200/convert.py and run by the CUDA engine gives torch's own logits for the same input, top-1 identical.
    torch = pytest.importorskip("torch")
    torchvision = pytest.importorskip("torchvision")
    from shadernn_b200 import convert
    torch.manual_seed(11)
    model = getattr(torchvision.models, name)(weights=None, num_classes=37)
    g = torch.Generator().manual_seed(12)
    for m in model.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.weight.data.uniform_(0.5, 1.5, generator=g)
            m.bias.data.uniform_(-0.1, 0.1, generator=g)
            m.running_mean.uniform_(-0.1, 0.1, generator=g)
            m.running_var.uniform_(0.5, 1.5, generator=g)
    model.eval()
    path = str(tmp_path / (name + ".json"))
    convert.export(model, path, input_hw=(96, 96), split=True)
    x = np.random.default_rng(4).uniform(-1, 1, (5, 96, 96, 3)).astype(np.float32)
    with torch.no_grad():
        want = model(torch.from_numpy(x).permute(0, 3, 1, 2).contiguous()).numpy()
    m = core.MixedInferenceCore(ctx, path, batch=5, fuse=True, use_cuda_graph=True)
    out, cls = m.run(x)
    got = out.reshape(5, -1)
    scale = float(np.abs(want).max())
    assert float(np.abs(got - want).max()) <= EPS * scale, (float(np.abs(got - want).max()), scale)
    assert np.array_equal(cls - 1, want.argmax(1))


def test_dump_outputs_diff_against_oracle_dumps(ctx, model_dir, tmp_path):
    # the --dump_outputs workflow (vulkanBackend.cpp:108-143): every layer's output as a reference-format .dump file, diffed
    # with tools/compare_dumps.py's machinery against dumps of the ground truth (here the oracle; elsewhere a ShaderNN/ncnn run)
    from shadernn_b200 import dumpio
    path, layers = modelzoo.build("resnet18", model_dir, input_hw=(64, 64))
    x = modelzoo.synthetic_input("resnet18", 2, (64, 64))
    want = oracle.Model(path).run(x, return_all=True)
    m = core.MixedInferenceCore(ctx, path, batch=2, input_hw=(64, 64), fuse=False)
    m.run(x)
    got_dir, ref_dir = tmp_path / "got", tmp_path / "ref"
    got_dir.mkdir(), ref_dir.mkdir()
    m.dump_outputs(str(got_dir))
    files = set(os.listdir(got_dir))
    expected = set()
    for i in range(m.num_layers):
        lname, _, _ = m.layer_info(i)
        for n in range(2):
            fname = "%s pass[0].dump.n%d" % (lname, n)
            expected.add(fname)
            dumpio.write_dump(str(ref_dir / fname), want[i][n])
    assert files == expected, (sorted(files - expected)[:3], sorted(expected - files)[:3])
    # the tool's default tolerance is the reference's own (0.01 abs-and-rel, testutil.cpp:351-361); the strict per-layer check at
    # 1e-3 relative to each tensor's range is layerwise_check above
    rows = dumpio.compare_dirs(str(got_dir), str(ref_dir), eps=0.01)
    assert len(rows) == 2 * m.num_layers and all(r[4] == "ok" for r in rows), [r for r in rows if r[4] != "ok"][:3]


@pytest.mark.parametrize("h,w,c,k,oc,padding,prepad", [
    (37, 53, 3, 7, 64, "same", None),          # the ResNet stem's shape class, ragged size
    (64, 301, 3, 3, 32, "valid", (0, 1, 0, 1)),  # MobileNetV2's: explicit (0,1) padding folded into the convolution
    (40, 531, 4, 5, 16, "same", None),         # three 128-pixel tiles per output row, 4 channels
    (33, 45, 1, 3, 24, "same", None),          # 1 channel
    (30, 41, 2, 9, 48, "same", None),          # 9 taps: three K steps per filter row
])
def test_stem_feed_mode_shapes(ctx, tmp_path, h, w, c, k, oc, padding, prepad):
    # conv_rowwin_kernel's feed mode (stride-2 convolutions with <= 4 input channels reading a model input: the compact 4-channel
    # copy written by the input kernels) against the oracle, fp32 and 8-bit input paths, fused and unfused
    b = modelzoo.Builder(7)
    x = b.input(w, h, c)
    if prepad:
        x = b.pad(x, *prepad)
    x = b.conv(x, oc, k, 2, padding, "relu", bias=True)
    b.conv(x, 8, 1, 1, "valid", "linear", bias=True)
    path = str(tmp_path / "stem.json")
    modelzoo.write_model(b.layers, path)
    rng = np.random.default_rng(3)
    img = rng.uniform(-1, 1, (3, h, w, c)).astype(np.float32)
    want = oracle.Model(path).run(img, return_all=True)
    conv_id = 2 if prepad else 1
    for fuse in (False, True):
        m = core.MixedInferenceCore(ctx, path, batch=3, fuse=fuse, use_cuda_graph=fuse)
        m.set_input(img)
        m.forward()
        ctx.sync()
        if not (prepad and not fuse):  # unfused, the Pad layer's output (not a model input) feeds the convolution: regular path
            m.time_layers()
            assert m.layer_kernel(conv_id) == "conv_rowwin_kernel<feed>", m.layer_kernel(conv_id)
        assert_layer_close(m.layer_output(conv_id), want[conv_id], EPS, "stem conv fuse=%d" % fuse)
        assert_layer_close(m.get_output(), want[-1], EPS, "head fuse=%d" % fuse)
    # 8-bit images normalised on the device take the same feed (split_u8_kernel writes it)
    if c in (3, 4):
        u8 = rng.integers(0, 256, (3, h, w, c), dtype=np.uint8)
        mean, norm = [127.5] * 4, [1 / 127.5] * 4
        xf = (u8.astype(np.float32) - 127.5) * np.float32(1 / 127.5)
        want8 = oracle.Model(path).run(xf)
        m = core.MixedInferenceCore(ctx, path, batch=3, fuse=True, use_cuda_graph=True)
        got8, _ = m.run_u8(u8, mean, norm, want_classes=False)
        assert_layer_close(got8, want8.reshape(got8.shape), EPS, "u8 input")


def test_repeated_loads_and_first_launches(ctx, model_dir):
    # Regression test of a start-up race of the halo convolution (pre-issued weight stages waited for after the MMA thread had released
    # them): it only showed on FIRST launches, when the producer warp was slow (cold instruction cache) - so load, run once, drop, repeat.
    path, _ = modelzoo.build("resnet18", model_dir, input_hw=(224, 224))
    x = modelzoo.synthetic_input("resnet18", 32, (224, 224))
    ref = {}
    for i in range(6):
        m = core.MixedInferenceCore(ctx, path, batch=32, fuse=bool(i & 1), use_cuda_graph=bool(i & 1))
        m.set_input(x)
        m.forward()
        out = m.get_output()
        assert np.array_equal(out, ref.setdefault(i & 1, out)), i  # every load of a mode computes the same bits
        del m
