"""The committed fixtures of the reference's candy-9_simplified.onnx (generator tests/golden/make_candy_golden.py):
 * tests/golden/candy_head_golden.npz as an ONNX-style graph dict for shadernn_b200/onnx2snn.convert_graph: the first two
   stages with their real weights;
 * tests/golden/candy_graph_golden.npz written back out as a whole ONNX file (whole_model_onnx)."""
import os

import numpy as np

from shadernn_b200 import onnx2snn

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "candy_head_golden.npz")
GRAPH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "candy_graph_golden.npz")


def head_graph():
    z = np.load(GOLDEN)
    init = {k[5:]: z[k] for k in z.files if k.startswith("init/")}
    ops = [str(o) for o in z["node_ops"]]
    assert ops == ["Pad", "Conv", "InstanceNormalization", "Relu", "Pad", "Conv", "InstanceNormalization", "Relu"]
    names = sorted(init)  # conv1.conv2d.{bias,weight}, conv2.conv2d.{bias,weight}, in1.{bias,weight}, in2.{bias,weight}
    nodes, t = [], "input1"
    for s, (k, st, p) in enumerate([(9, 1, 4), (3, 2, 1)], start=1):
        nodes.append({"op": "Pad", "input": [t], "output": ["p%d" % s], "name": "pad%d" % s, "attr": {"mode": "reflect", "pads": [0, 0, p, p, 0, 0, p, p]}})
        nodes.append({"op": "Conv", "input": ["p%d" % s, "conv%d.conv2d.weight" % s, "conv%d.conv2d.bias" % s], "output": ["c%d" % s], "name": "conv%d" % s,
                      "attr": {"kernel_shape": [k, k], "strides": [st, st], "pads": [0, 0, 0, 0], "group": 1}})
        nodes.append({"op": "InstanceNormalization", "input": ["c%d" % s, "in%d.weight" % s, "in%d.bias" % s], "output": ["n%d" % s], "name": "in%d" % s,
                      "attr": {"epsilon": 1e-5}})
        nodes.append({"op": "Relu", "input": ["n%d" % s], "output": ["r%d" % s], "name": "relu%d" % s, "attr": {}})
        t = "r%d" % s
    assert all(n in names for nd in nodes for n in nd["input"][1:])
    return {"nodes": nodes, "init": init, "inputs": [("input1", [1, 3, 64, 64])], "outputs": [(t, [])]}, z["x"], z["y"]


def varint(v):
    out = b""
    v &= (1 << 64) - 1
    while True:
        b = v & 0x7F
        v >>= 7
        out += bytes([b | (0x80 if v else 0)])
        if not v:
            return out


def field(f, w, v):
    """Encode one protobuf field as onnx2snn._fields yields it: (field number, wire type, value)."""
    key = varint((f << 3) | w)
    if w == 0:
        return key + varint(v)
    if w == 2:
        return key + varint(len(v)) + bytes(v)
    return key + bytes(v)  # wire types 1 and 5: the fixed 8 or 4 bytes


def whole_model_onnx(path):
    """Write the whole candy-9_simplified.onnx to `path` and return it. The file is the reference's byte for byte (every node,
    attribute, value info and 1-D initialiser as exported) except the 16 convolution kernels, 1.67 M of the model's 1.68 M
    weights, which the fixture does not hold: each is filled with seeded normal values of the real kernel's mean and
    standard deviation."""
    z = np.load(GRAPH)
    rng = np.random.default_rng(0)

    def tensor(b):
        dims, name = [], ""
        for f, w, v in onnx2snn._fields(b):
            if f == 1:
                dims += onnx2snn._ints(w, v)
            elif f == 8:
                name = bytes(v).decode()
        if "stats/" + name not in z.files:
            return bytes(b)
        mean, std = z["stats/" + name]
        return bytes(b) + field(9, 2, (rng.standard_normal(int(np.prod(dims))) * std + mean).astype("<f4").tobytes())

    def graph(b):
        return b"".join(field(f, w, tensor(v) if f == 5 else v) for f, w, v in onnx2snn._fields(b))

    model = b"".join(field(f, w, graph(v) if f == 7 else v) for f, w, v in onnx2snn._fields(memoryview(z["onnx"].tobytes())))
    with open(path, "wb") as f:
        f.write(model)
    return path
