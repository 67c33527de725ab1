"""GPU tests of the folded projection shortcut (fusion pass (5) of MixedInferenceCore::init): in a down-sampling block
Add(conv3x3(y), conv1x1_s2(x)) the 1x1 projection runs as extra K blocks of the 3x3 convolution's implicit GEMM. Checked on
Builder-made blocks against the oracle, against the same model with fuse=0, and against the unfolded fused form
(SNNB_NO_SHORTCUT_FOLD=1): one launch less per block, the hidden convolutions refuse layer_output, results unchanged."""
import os

import numpy as np
import pytest

from oracle import oracle
from shadernn_b200 import core, modelzoo
from shadernn_b200._lib import SnnbError

pytestmark = pytest.mark.gpu

# (input h, w, block input channels, block output channels)
SHAPES = {
    "56to28": (56, 56, 64, 128),
    "28to14": (28, 28, 128, 256),
    "14to7": (14, 14, 256, 512),    # the split-K layer of ResNet-18
    "ragged13x9": (26, 18, 64, 128),
    "ic24oc40": (16, 16, 24, 40),   # channel counts that are not multiples of 64
}


def block(path, shape, order="ds_first", ds_act="linear", ds_k=1, ds_reader=False):
    """pre-conv -> [conv3x3 s2 + relu -> conv3x3 (c2)] + projection (ds) -> Add + relu, BN on every conv (folded at load)."""
    h, w, ic, oc = shape
    b = modelzoo.Builder()
    x = b.input(w, h, ic)
    x = b.conv(x, ic, 3, 1, "same", "relu", bias=True, bn=True)
    y = b.conv(x, oc, 3, 2, "same", "relu", bias=True, bn=True)
    y = b.conv(y, oc, 3, 1, "same", "linear", bias=True, bn=True, gain=0.5)
    s = b.conv(x, oc, ds_k, 2, "valid" if ds_k == 1 else "same", ds_act, bias=True, bn=True, gain=1.0)
    a = b.add(s, y, "relu") if order == "ds_first" else b.add(y, s, "relu")
    if ds_reader:
        b.add(a, s, "linear")  # a second reader of the projection's output
    return modelzoo.write_model(b.layers, path), b.layers, (y, s, a)


def load(ctx, path, batch, precision, fuse=True, graph=False, fold=True, algo="auto"):
    if not fold:
        os.environ["SNNB_NO_SHORTCUT_FOLD"] = "1"
    try:
        return core.MixedInferenceCore(ctx, path, batch=batch, fuse=fuse, use_cuda_graph=graph, precision=precision, conv_algo=algo)
    finally:
        os.environ.pop("SNNB_NO_SHORTCUT_FOLD", None)


def run(ctx, m, x, layer):
    m.set_input(x)
    m.forward()
    ctx.sync()
    return m.layer_output(layer)


def rel(got, want):
    return float(np.abs(got.astype(np.float64) - want).max() / max(float(np.abs(want).max()), 1e-30))


@pytest.mark.parametrize("name", list(SHAPES))
@pytest.mark.parametrize("batch", [1, 3, 32])
@pytest.mark.parametrize("precision", ["fp32x3", "fp16w", "fp16"])
@pytest.mark.parametrize("graph", [False, True])
def test_folded_block(ctx, tmp_path, name, batch, precision, graph):
    shape = SHAPES[name]
    path, layers, (c2, ds, add) = block(str(tmp_path / "block.json"), shape, order="ds_first" if batch != 3 else "c2_first")
    x = np.random.default_rng(batch).standard_normal((batch, shape[0], shape[1], shape[2])).astype(np.float32)
    fused = load(ctx, path, batch, precision, graph=graph)
    plain = load(ctx, path, batch, precision, fuse=False)
    nofold = load(ctx, path, batch, precision, fold=False)
    # fp16 storage at batch 32: the planner gives the 56x56 and 28x28 blocks' 3x3 convolution to the halo mode, which has no
    # shortcut operand - the fold declines and the block runs as before
    folds = not (precision == "fp16" and batch == 32 and name in ("56to28", "28to14"))
    assert fused.launches_per_forward == nofold.launches_per_forward - (1 if folds else 0)
    got = run(ctx, fused, x, add)
    ref = run(ctx, plain, x, add)
    # fp16 storage rounds the unfused projection's output to fp16 before the add; the fold keeps it in the fp32 accumulator
    assert rel(got, ref) <= (1e-4 if precision != "fp16" else 2e-3), (rel(got, ref), name, batch, precision)
    if precision == "fp32x3":
        n = min(batch, 3)
        want = oracle.Model(path).run(x[:n], return_all=True)[add]
        assert rel(got[:n], want) <= 3e-4, rel(got[:n], want)
    fused.time_layers()
    if folds:
        assert fused.layer_kernel(ds) == ""
        assert fused.layer_kernel(c2).startswith("conv_umma_kernel") and "halo" not in fused.layer_kernel(c2), fused.layer_kernel(c2)
        for hidden in (c2, ds):
            with pytest.raises(SnnbError, match="fuse=0"):
                fused.layer_output(hidden)
    else:
        assert fused.layer_kernel(ds).startswith("conv_umma_kernel")


@pytest.mark.parametrize("case", ["ds_relu", "ds_second_reader", "ds_3x3", "simt"])
def test_fold_declines(ctx, tmp_path, case):
    shape = SHAPES["28to14"]
    path, layers, (c2, ds, add) = block(str(tmp_path / "block.json"), shape, ds_act="relu" if case == "ds_relu" else "linear",
                                        ds_k=3 if case == "ds_3x3" else 1, ds_reader=case == "ds_second_reader")
    algo = "simt" if case == "simt" else "auto"
    x = np.random.default_rng(0).standard_normal((2, shape[0], shape[1], shape[2])).astype(np.float32)
    fused = load(ctx, path, 2, "fp32x3", algo=algo)
    nofold = load(ctx, path, 2, "fp32x3", fold=False, algo=algo)
    assert fused.launches_per_forward == nofold.launches_per_forward
    got = run(ctx, fused, x, len(layers) - 1)
    want = oracle.Model(path).run(x, return_all=True)[len(layers) - 1]
    assert rel(got, want) <= 3e-4
    fused.time_layers()
    assert fused.layer_kernel(ds) != ""  # the projection keeps its own launch
