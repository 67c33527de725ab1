"""Generator of tests/golden/candy_head_golden.npz and tests/golden/candy_graph_golden.npz from a reference checkout:

    python tests/golden/make_candy_golden.py <reference checkout>/modelzoo/StyleTransfer/candy-9_simplified.onnx

The only real-weight model in the reference checkout is modelzoo/StyleTransfer/candy-9_simplified.onnx. At 6.7 MB it is not
part of this repository, so this script freezes two fixtures of it:
 * candy_head_golden.npz: (a) the initialisers of its first two stages (reflect-pad + 9x9 conv 3->32 + InstanceNorm + ReLU;
   reflect-pad + 3x3 stride-2 conv 32->64 + InstanceNorm + ReLU: ~105 KB of fp32), (b) a 64x64 input in the model's own range
   [0, 255], and (c) what torch computes for those ONNX nodes (shadernn_b200/onnx2snn.torch_eval on the truncated graph, i.e.
   the ONNX semantics themselves, no conversion involved). tests/ rebuild the SNN model from (a) with the converter and hold
   the oracle and the CUDA engine to (c).
 * candy_graph_golden.npz: the ONNX file's bytes without the raw data of the convolution kernels (every node, attribute and
   1-D initialiser kept as exported), plus each kernel's mean and standard deviation. tests/_candy_fixture.whole_model_onnx
   writes it back out as a whole ONNX file with seeded kernels of those statistics, on which tests/ hold the converter, the
   oracle and the CUDA engine to torch's evaluation of the whole graph.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
from shadernn_b200 import modelzoo, onnx2snn  # noqa: E402
from _candy_fixture import field  # noqa: E402

HEAD_NODES = 8  # Pad Conv IN Relu Pad Conv IN Relu


def truncated(g, n_nodes):
    nodes = g["nodes"][:n_nodes]
    used = {t for nd in nodes for t in nd["input"]}
    return {"nodes": nodes, "init": {k: v for k, v in g["init"].items() if k in used}, "inputs": g["inputs"], "outputs": [(nodes[-1]["output"][0], [])]}


def head(src):
    g = onnx2snn.load_onnx(src)
    h = truncated(g, HEAD_NODES)
    x = modelzoo.synthetic_input("candy", 1, (64, 64))
    y = onnx2snn.torch_eval(h, x)
    out = {"x": x, "y": y, "node_ops": np.array([nd["op"] for nd in h["nodes"]])}
    for k, v in h["init"].items():
        out["init/" + k] = np.array(v)
    path = os.path.join(HERE, "candy_head_golden.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes; output", y.shape, "max", float(np.abs(y).max()))


def graph(src):
    stats = {}

    def tensor(b):
        name, a = onnx2snn._tensor(b)
        if a.ndim < 2:
            return bytes(b)
        stats["stats/" + name] = np.array([a.mean(dtype=np.float64), a.std(dtype=np.float64)])
        return b"".join(field(f, w, v) for f, w, v in onnx2snn._fields(b) if f != 9)  # TensorProto.raw_data = 9

    def graph_of(b):
        return b"".join(field(f, w, tensor(v) if f == 5 else v) for f, w, v in onnx2snn._fields(b))

    with open(src, "rb") as f:
        raw = f.read()
    # the encoder must reproduce the exporter's bytes, or the fixture would not be the reference's file
    assert b"".join(field(f, w, v) for f, w, v in onnx2snn._fields(memoryview(raw))) == raw
    skeleton = b"".join(field(f, w, graph_of(v) if f == 7 else v) for f, w, v in onnx2snn._fields(memoryview(raw)))
    path = os.path.join(HERE, "candy_graph_golden.npz")
    np.savez_compressed(path, onnx=np.frombuffer(skeleton, np.uint8), **stats)
    print(path, os.path.getsize(path), "bytes;", len(stats), "kernels replaced by their statistics")


if __name__ == "__main__":
    head(sys.argv[1])
    graph(sys.argv[1])
