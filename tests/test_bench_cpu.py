"""bench.py --dump-outputs without a GPU: file names, dtype, and the fixed sample that keeps a large dump under its cap, on a
stand-in for the engine's model."""
import os
import types

import numpy as np

import bench


class _Model:
    def __init__(self, outs):
        self.outs = outs
        self.num_outputs = len(outs)

    def get_output(self, i):
        return self.outs[i].copy()


def _workload(outs):
    return types.SimpleNamespace(model=_Model(outs), detector=False, layers=[])


def test_dump_outputs_writes_every_output(tmp_path):
    rng = np.random.default_rng(1)
    outs = [rng.standard_normal((2, 1, 1, 10)).astype(np.float32), rng.standard_normal((2, 4, 4, 3)).astype(np.float32)]
    bench.dump_outputs(_workload(outs), str(tmp_path / "d"))
    assert sorted(os.listdir(tmp_path / "d")) == ["output_0.npy", "output_1.npy"]
    for i, o in enumerate(outs):
        got = np.load(tmp_path / "d" / ("output_%d.npy" % i))
        assert got.dtype == np.float32 and np.array_equal(got, o)


def test_dump_outputs_samples_above_the_cap(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 4000)
    # element values = flat positions (negated in the second output), so a sample shows which positions it kept
    outs = [np.arange(3000, dtype=np.float32).reshape(1, 10, 100, 3), -np.arange(1000, dtype=np.float32).reshape(1, 1, 1, 1000)]
    for d in ("a", "b"):
        bench.dump_outputs(_workload(outs), str(tmp_path / d))
    total = 0
    for i, o in enumerate(outs):
        a, b = (np.load(tmp_path / d / ("output_%d.npy" % i)) for d in ("a", "b"))
        assert a.dtype == np.float32 and np.array_equal(a, b)  # the same sample from run to run
        assert a.ndim == 1 and np.all(np.diff(np.abs(a)) > 0) and np.isin(a, o).all()  # distinct positions, ascending
        total += a.nbytes
    assert 2000 < total <= 4000
