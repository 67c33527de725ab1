"""ONNX -> ShaderNN JSON converter (shadernn_b200/onnx2snn.py, SURVEY §8 f-N1): the hand-rolled protobuf reader, the
conversion rules, and — the one reference-held pin the conv path has — modelzoo/StyleTransfer/candy-9_simplified.onnx: the
converted model, walked by the oracle, must reproduce what torch computes for the ONNX graph itself. Two committed fixtures
(generator tests/golden/make_candy_golden.py) stand in for the 6.7 MB file: candy_head_golden.npz carries the first two
stages' real initialisers and torch's outputs; candy_graph_golden.npz the whole file except the convolution kernels' values."""
import os
import struct

import numpy as np

from oracle import oracle
from shadernn_b200 import modelzoo, onnx2snn

from _candy_fixture import head_graph as _head_graph
from _candy_fixture import varint as _vi
from _candy_fixture import whole_model_onnx

HERE = os.path.dirname(os.path.abspath(__file__))


# ---- a minimal protobuf ENCODER, test-side only, to feed the reader with hand-made messages -------------------------
def _ld(field, payload):
    return _vi((field << 3) | 2) + _vi(len(payload)) + payload


def _int(field, v):
    return _vi((field << 3) | 0) + _vi(v)


def _tensor(name, arr):
    arr = np.asarray(arr)
    dt = {np.dtype("float32"): 1, np.dtype("int64"): 7}[arr.dtype]
    return b"".join(_int(1, d) for d in arr.shape) + _int(2, dt) + _ld(8, name.encode()) + _ld(9, arr.tobytes())


def _attr_ints(name, ints):
    return _ld(1, name.encode()) + b"".join(_int(8, i) for i in ints)


def _attr_packed_ints(name, ints):
    return _ld(1, name.encode()) + _ld(8, b"".join(_vi(i) for i in ints))


def _attr_f(name, f):
    return _ld(1, name.encode()) + _vi((2 << 3) | 5) + struct.pack("<f", f)


def _attr_s(name, s):
    return _ld(1, name.encode()) + _ld(4, s.encode())


def _node(op, ins, outs, attrs=(), name=""):
    return b"".join(_ld(1, i.encode()) for i in ins) + b"".join(_ld(2, o.encode()) for o in outs) + _ld(3, name.encode()) + _ld(4, op.encode()) + b"".join(
        _ld(5, a) for a in attrs)


def _value_info(name, dims):
    shape = b"".join(_ld(1, _int(1, d)) for d in dims)
    return _ld(1, name.encode()) + _ld(2, _ld(1, _int(1, 1) + _ld(2, shape)))


def _model(nodes, inits, inp, out):
    graph = b"".join(_ld(1, n) for n in nodes) + b"".join(_ld(5, t) for t in inits) + _ld(11, inp) + _ld(12, out)
    return _int(1, 4) + _ld(7, graph)


def test_reader_parses_hand_made_model(tmp_path):
    rng = np.random.default_rng(1)
    w = rng.standard_normal((8, 3, 3, 3)).astype(np.float32)
    b = rng.standard_normal(8).astype(np.float32)
    g_, be, mu, var = (rng.uniform(0.5, 1.5, 8).astype(np.float32) for _ in range(4))
    nodes = [
        _node("Pad", ["x"], ["p"], [_attr_s("mode", "reflect"), _attr_ints("pads", [0, 0, 1, 1, 0, 0, 1, 1])], "pad0"),
        _node("Conv", ["p", "w", "b"], ["c"], [_attr_packed_ints("kernel_shape", [3, 3]), _attr_ints("strides", [1, 1]), _attr_ints("pads", [0, 0, 0, 0]),
                                                _attr_ints("group", []) + _int(3, 1)], "conv0"),
        _node("BatchNormalization", ["c", "g", "be", "mu", "var"], ["n"], [_attr_f("epsilon", 1e-5)], "bn0"),
        _node("LeakyRelu", ["n"], ["y"], [_attr_f("alpha", 0.2)], "act0"),
    ]
    inits = [_tensor("w", w), _tensor("b", b), _tensor("g", g_), _tensor("be", be), _tensor("mu", mu), _tensor("var", var)]
    path = tmp_path / "tiny.onnx"
    path.write_bytes(_model(nodes, inits, _value_info("x", [1, 3, 16, 16]), _value_info("y", [1, 8, 16, 16])))
    g = onnx2snn.load_onnx(str(path))
    assert [n["op"] for n in g["nodes"]] == ["Pad", "Conv", "BatchNormalization", "LeakyRelu"]
    assert g["inputs"] == [("x", [1, 3, 16, 16])] and g["nodes"][1]["attr"]["kernel_shape"] == [3, 3]
    assert np.array_equal(g["init"]["w"], w) and abs(g["nodes"][3]["attr"]["alpha"] - 0.2) < 1e-7 and g["nodes"][0]["attr"]["mode"] == "reflect"
    # conversion: the Pad folds into the conv, BN and the activation merge into it (one Conv2D layer besides the input)
    jpath, layers = onnx2snn.convert(str(path), str(tmp_path), split=False)
    assert [l["type"] for l in layers] == ["InputLayer", "Conv2D"]
    L = layers[1]
    assert L["padding"] == [[1, 1], [1, 1]] and L["mode"] == "reflect" and L["activation"] == "leakyRelu" and L["useBatchNormalization"] == "True"
    x = rng.uniform(-1, 1, (2, 16, 16, 3)).astype(np.float32)
    want = onnx2snn.torch_eval(g, x)
    got = oracle.Model(jpath).run(x)
    assert float(np.abs(got - want).max()) <= 2e-5 * float(np.abs(want).max())
    # the tool's literal output (standalone Pad layer) is available too
    _, layers2 = onnx2snn.convert(str(path), str(tmp_path / "nofold"), split=False, fold_pads=False)
    assert [l["type"] for l in layers2] == ["InputLayer", "Pad", "Conv2D"] and layers2[1]["pads"] == [0, 0, 1, 1, 0, 0, 1, 1]


def test_real_candy_weights_head_matches_torch_golden(tmp_path):
    # reference-held weights, torch-held expectation (generated from the ONNX file by tests/golden/make_candy_golden.py)
    g, x, want = _head_graph()
    layers = onnx2snn.convert_graph(g, input_hw=(64, 64))
    assert [l["type"] for l in layers] == ["InputLayer", "Conv2D", "InstanceNormalization", "Conv2D", "InstanceNormalization"]
    path = modelzoo.write_model(layers, str(tmp_path / "candy_head_layers.json"), split=True)
    got = oracle.Model(path).run(x)
    assert got.shape == want.shape
    assert float(np.abs(got - want).max()) <= 5e-5 * float(np.abs(want).max())


def test_whole_candy_model_from_the_reference_checkout(tmp_path):
    # the reference's file as the fixture holds it: its own graph and encoding, seeded convolution kernels (_candy_fixture)
    src = whole_model_onnx(str(tmp_path / "candy-9_simplified.onnx"))
    g = onnx2snn.load_onnx(src)
    assert len(g["nodes"]) == 64 and len(g["init"]) == 64
    path, layers = onnx2snn.convert(src, str(tmp_path), input_hw=(96, 96))
    assert os.path.basename(path) == "candy-9_simplified_layers.json" and os.path.exists(str(tmp_path / "candy-9_simplified_weights.bin"))  # onnxToJsonConverter.py:69-73
    assert len(layers) == 39 and sum(l["type"] == "Conv2D" for l in layers) == 16 and sum(l["type"] == "InstanceNormalization" for l in layers) == 15
    x = modelzoo.synthetic_input("candy", 1, (96, 96))
    want = onnx2snn.torch_eval(g, x)
    got = oracle.Model(path).run(x)
    assert float(np.abs(got - want).max()) <= 5e-5 * float(np.abs(want).max())
