"""Generate tests/golden/ref_cpu_golden.npz and tests/golden/ref_cpu_live_golden.npz from the REFERENCE ITSELF
(oracle/_ref/libsnn_ref.so = the reference's core/src/ic2/cpulayer.h + demo/common/prng.h, compiled where they lie in a
reference checkout).

The reference is not part of this repository, so its outputs are committed here as small fixtures and this script is the
recipe that produced them:   make -C oracle ref REF=<reference checkout> && python tests/golden/make_golden.py
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle  # noqa: E402


def main():
    r = oracle.ref()
    assert r is not None, "build oracle/_ref first (needs /root/reference)"
    out = {}
    # --- prng.h: seed 7767517 (convolutionTest.cpp:417) ---
    r.ref_srand(C.c_uint64(7767517))
    out["prng_u64"] = np.array([r.ref_rand_u64() for _ in range(256)], dtype=np.uint64)
    r.ref_srand(C.c_uint64(7767517))
    out["prng_float"] = np.array([r.ref_random_float(-1.2, 1.2) for _ in range(256)], dtype=np.float32)
    r.ref_srand(C.c_uint64(1))
    out["prng_u64_seed1"] = np.array([r.ref_rand_u64() for _ in range(64)], dtype=np.uint64)

    # --- cpulayer.h Dense + activation: the reference's dense test grid 11 -> 5 (denseTest.cpp:111) and a few more ---
    rng = np.random.default_rng(7767517)
    cases = []
    for (n_in, n_out) in [(11, 5), (3, 2), (512, 10), (64, 33)]:
        for act, alpha in [("", 0.0), ("relu", 0.0), ("leakyRelu", 0.1), ("sigmoid", 0.0), ("tanh", 0.0), ("softmax", 0.0), ("SiLU", 0.0)]:
            x = rng.uniform(-2, 2, n_in).astype(np.float32)
            k = rng.uniform(-1.2, 1.2, (n_out, n_in)).astype(np.float32)
            b = rng.uniform(-0.5, 0.5, n_out).astype(np.float32)
            y = np.empty(n_out, np.float32)
            rc = r.ref_dense(x.ctypes.data_as(C.c_void_p), n_in, k.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), n_out, act.encode(),
                             alpha, y.ctypes.data_as(C.c_void_p))
            assert rc == 0
            cases.append((n_in, n_out, act, alpha, x, k, b, y))
    out["dense_n"] = np.array(len(cases))
    for i, (n_in, n_out, act, alpha, x, k, b, y) in enumerate(cases):
        out["dense_%d_act" % i] = np.array(act)
        out["dense_%d_alpha" % i] = np.array(alpha, np.float32)
        out["dense_%d_x" % i] = x
        out["dense_%d_k" % i] = k
        out["dense_%d_b" % i] = b
        out["dense_%d_y" % i] = y
    # the survey's smoke value: Dense 3->2 + softmax gave 0.017986 0.982014 (SURVEY F5)
    x = np.array([1, 2, 3], np.float32)
    k = np.array([[1, 0, 0], [0, 1, 1]], np.float32)
    b = np.zeros(2, np.float32)
    y = np.empty(2, np.float32)
    r.ref_dense(x.ctypes.data_as(C.c_void_p), 3, k.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), 2, b"softmax", 0.0, y.ctypes.data_as(C.c_void_p))
    out["smoke_softmax"] = y
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_cpu_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, "smoke softmax:", y)


def live_cases():
    """The long PRNG streams and the Dense cases that tests/test_oracle_cpu.py holds the oracle to (the *_live_reference tests)."""
    r = oracle.ref()
    assert r is not None, "build oracle/_ref first (needs a reference checkout)"
    out = {}
    for seed in (7767517, 1, 123456789):
        r.ref_srand(C.c_uint64(seed))
        out["prng_u64_%d" % seed] = np.array([r.ref_rand_u64() for _ in range(3000)], dtype=np.uint64)  # crosses several 55-draw refills
    rng = np.random.default_rng(5)
    for act in ["", "relu", "leakyRelu", "sigmoid", "tanh", "softmax"]:
        x = rng.uniform(-2, 2, 37).astype(np.float32)
        k = rng.uniform(-1, 1, (9, 37)).astype(np.float32)
        b = rng.uniform(-1, 1, 9).astype(np.float32)
        y = np.empty(9, np.float32)
        assert r.ref_dense(x.ctypes.data_as(C.c_void_p), 37, k.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), 9, act.encode(), 0.2,
                           y.ctypes.data_as(C.c_void_p)) == 0
        for s, v in zip("xkby", (x, k, b, y)):
            out["dense_%s_%s" % (act or "linear", s)] = v
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_cpu_live_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path)


if __name__ == "__main__":
    main()
    live_cases()
