"""CPU suite (-m "not gpu"): pins the ORACLE.

 * against the reference itself: tests/golden/ref_cpu_golden.npz and ref_cpu_live_golden.npz were produced by the compiled
   reference code (cpulayer.h Dense/softmax/activations, prng.h) — see tests/golden/make_golden.py;
 * against hand-derived known answers built from the reference's own unit-test constructions (SURVEY §4, §8c):
   all-ones inputs reduce a conv to per-output-channel weight sums, BN with gamma=1 mu=0 var=1 beta=0 is a factor
   1/sqrt(1.001), pooling with sentinel values, the dims formulas of conv2d.cpp / maxpool2d.cpp.
The reference's numeric ground truth for Conv/Pool (ncnn 20211208) is not available offline: "parity vs ncnn unpinned".
"""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import oracle

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_cpu_golden.npz")
LIVE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_cpu_live_golden.npz")


@pytest.fixture(scope="module")
def gold(built):
    return np.load(GOLD)


def test_prng_matches_reference_golden(gold):
    oracle.srand(7767517)
    got = np.array([oracle.lib().orc_rand_u64() for _ in range(256)], dtype=np.uint64)
    assert np.array_equal(got, gold["prng_u64"])
    oracle.srand(7767517)
    gotf = np.array([oracle.lib().orc_random_float(-1.2, 1.2) for _ in range(256)], dtype=np.float32)
    assert np.array_equal(gotf, gold["prng_float"])  # bit-exact
    oracle.srand(1)
    got1 = np.array([oracle.lib().orc_rand_u64() for _ in range(64)], dtype=np.uint64)
    assert np.array_equal(got1, gold["prng_u64_seed1"])


def test_prng_matches_live_reference(built):
    # the reference library's own streams, recorded by tests/golden/make_golden.py (live_cases)
    live = np.load(LIVE)
    for seed in (7767517, 1, 123456789):
        oracle.srand(seed)
        a = [oracle.lib().orc_rand_u64() for _ in range(3000)]  # crosses several 55-draw refills
        b = live["prng_u64_%d" % seed].tolist()
        assert a == b


def test_dense_matches_reference_golden(gold):
    n = int(gold["dense_n"])
    assert n >= 20
    for i in range(n):
        act = str(gold["dense_%d_act" % i])
        alpha = float(gold["dense_%d_alpha" % i])
        x, k, b, y = (gold["dense_%d_%s" % (i, s)] for s in "xkby")
        got = oracle.dense(x.reshape(1, 1, 1, -1), k, b, act, alpha).ravel()
        # Eigen's blocked dot product vs a sequential sum: same fp32 arithmetic, different association
        # (error bound ~ n_in * eps32 * sum|w*x|; the 512-wide case reaches 1.3e-5 absolute on outputs of magnitude 35)
        tol = 4 * np.finfo(np.float32).eps * float(np.abs(k.astype(np.float64) * x).sum(axis=1).max()) + 1e-6
        assert np.allclose(got, y, rtol=2e-6, atol=tol), (i, act, np.abs(got - y).max(), tol)
    sm = oracle.dense(np.array([1, 2, 3], np.float32).reshape(1, 1, 1, 3), np.array([[1, 0, 0], [0, 1, 1]], np.float32), np.zeros(2, np.float32),
                      "softmax").ravel()
    assert np.allclose(sm, gold["smoke_softmax"], rtol=1e-6)
    assert np.allclose(sm, [0.017986, 0.982014], atol=1e-6)  # the value quoted in SURVEY F5


def test_dense_matches_live_reference(built):
    # inputs and the reference library's outputs, recorded by tests/golden/make_golden.py (live_cases)
    live = np.load(LIVE)
    for act in ["", "relu", "leakyRelu", "sigmoid", "tanh", "softmax"]:
        x, k, b, y = (live["dense_%s_%s" % (act or "linear", s)] for s in "xkby")
        got = oracle.dense(x.reshape(1, 1, 1, -1), k, b, act, 0.2).ravel()
        assert np.allclose(got, y, rtol=2e-6, atol=2e-6), act


# ---- known answers from the reference's own test constructions ----
def test_conv_all_ones_input_reduces_to_weight_sums(built):
    # convolutionTest.cpp:42-167: input all ones, weights RandomMat U[-1.2,1.2] from SRAND(7767517), bias 0,
    # BN gamma=1 mean=0 var=1 beta=0 -> y[oc] = sum(w[oc]) / sqrt(1.001) wherever the window is fully inside.
    oracle.srand(7767517)
    H = W = 8
    IC, OC, k = 16, 4, 3
    w = oracle.random_mat((OC, IC, k, k))
    x = np.ones((1, H, W, IC), np.float32)
    bn = {"gamma": np.ones(OC), "beta": np.zeros(OC), "mean": np.zeros(OC), "var": np.ones(OC)}
    o = oracle.same_padding(k, True)
    assert o == [1, 1, 1, 1]
    oh = oracle.conv_out_dim(H, k, 1, o[0], o[1])
    assert oh == 8
    y = oracle.conv2d(x, w, None, bn, 1, o[0], o[2], "constant", "", 0.0, (oh, oh))
    want = w.astype(np.float64).sum(axis=(1, 2, 3)) / np.sqrt(1.001)
    assert np.allclose(y[0, 3, 3], want, rtol=1e-5, atol=1e-5)
    # corner: only the 2x2 in-range taps contribute (constant padding reads 0)
    want_c = w[:, :, 1:, 1:].astype(np.float64).sum(axis=(1, 2, 3)) / np.sqrt(1.001)
    assert np.allclose(y[0, 0, 0], want_c, rtol=1e-5, atol=1e-5)
    # relu epilogue
    yr = oracle.conv2d(x, w, None, bn, 1, 1, 1, "constant", "relu", 0.0, (oh, oh))
    assert np.array_equal(yr, np.maximum(y, 0))


def test_conv_padding_modes(built):
    x = np.arange(1 * 4 * 5 * 1, dtype=np.float32).reshape(1, 4, 5, 1)
    w = np.zeros((1, 1, 3, 3), np.float32)
    w[0, 0, 0, 0] = 1.0  # picks the top-left tap: y[oy,ox] = x[oy-1, ox-1]
    yc = oracle.conv2d(x, w, None, None, 1, 1, 1, "constant", "", 0, (4, 5))
    yr = oracle.conv2d(x, w, None, None, 1, 1, 1, "replicate", "", 0, (4, 5))
    yf = oracle.conv2d(x, w, None, None, 1, 1, 1, "reflect", "", 0, (4, 5))
    assert yc[0, 0, 0, 0] == 0 and yc[0, 1, 1, 0] == x[0, 0, 0, 0]
    assert yr[0, 0, 0, 0] == x[0, 0, 0, 0] and yr[0, 0, 3, 0] == x[0, 0, 2, 0]
    assert yf[0, 0, 0, 0] == x[0, 1, 1, 0]  # reflect: -1 -> 1 (vk_conv2d.comp:176-179)


def test_dims_rules(built):
    # conv2d.cpp:102-113 (float then truncation) and conv2d.cpp:57-65 (even k: top/left = k/2-1)
    assert oracle.conv_out_dim(224, 7, 2, 3, 3) == 112
    assert oracle.conv_out_dim(112, 3, 2, 1, 1) == 56
    assert oracle.conv_out_dim(56, 1, 2, 0, 0) == 28
    assert oracle.conv_out_dim(8, 1, 1, 0, 0) == 8
    assert oracle.same_padding(4, True) == [1, 2, 1, 2]
    assert oracle.conv_out_dim(9, 4, 2, 1, 2) == 4  # even k: 9/2 + max(0, 1 + (pT+pB-1-k)/s = 0) = 4.5 -> 4
    # negative translations are clamped at 0 (std::max from 0, genericlayer.cpp:66-75): "valid" convs keep their size
    assert oracle.conv_out_dim(8, 4, 1, 1, 2) == 8
    assert oracle.conv_out_dim(10, 3, 1, 0, 0) == 10
    assert oracle.conv_out_dim(225, 3, 2, 0, 0) == 112  # MobileNetV2: Pad((0,1),(0,1)) + valid 3x3 s2
    assert oracle.same_padding(1, True) == [0, 0, 0, 0]
    assert oracle.same_padding(5, False) == [0, 0, 0, 0]
    # pools: maxpool2d.cpp:26-35
    assert oracle.pool_out_dim(112, 3, 2, False) == 56  # "same": floor(W/s + 1 - 1/s)
    assert oracle.pool_out_dim(9, 2, 3, False) == 3     # the reference's pooling grid (poolingTest.cpp:42-44)
    assert oracle.pool_out_dim(416, 2, 2, True) == 208
    assert oracle.pool_out_dim(13, 2, 1, False) == 13   # yolo's last pool: 2x2 s1 same
    assert oracle.pool_out_dim(7, 7, 7, True) == 1      # global pool: the avg reader defaults stride to the pool size
    assert oracle.pool_out_dim(7, 7, 1, True) == 7      # ... an explicit stride 1 would NOT collapse (translation clamped at 0)
    # depthwise: separableconvolution.cpp:77-86
    assert oracle.depthwise_out_dim(112, 3, 1, 1, 1) == 112
    assert oracle.depthwise_out_dim(113, 3, 2, 0, 0) == 56


def test_pooling_sentinels(built):
    # poolingTest.cpp:42-44,104: 9x9x4 input, k=2 s=3 'same' -> 3x3; avg divides by the number of VALID taps and the
    # window is never padded top/left (maxpool2dVulkan.cpp:57-60).
    x = np.full((1, 9, 9, 4), 100.0, np.float32)
    x[0, ::3, ::3, :] = 200.0
    oh = oracle.pool_out_dim(9, 2, 3, False)
    ya = oracle.pool2d(x, 2, 3, True, (oh, oh))
    ym = oracle.pool2d(x, 2, 3, False, (oh, oh))
    assert np.allclose(ya, (200 + 3 * 100) / 4.0)
    assert np.allclose(ym, 200.0)
    # clipped window at the bottom/right edge: 5x5 input, k=3 s=2 -> origin 4 holds one valid tap
    x2 = np.arange(25, dtype=np.float32).reshape(1, 5, 5, 1)
    o2 = oracle.pool_out_dim(5, 3, 2, False)
    assert o2 == 3
    y2 = oracle.pool2d(x2, 3, 2, True, (o2, o2))
    assert y2[0, 2, 2, 0] == 24.0
    assert y2[0, 0, 2, 0] == np.mean([4, 9, 14])
    ymax = oracle.pool2d(-x2 - 200000, 3, 2, False, (o2, o2))
    assert ymax[0, 0, 0, 0] == -100000.0  # init value wins over very negative inputs (vk_maxpool2d.comp:53)


def test_batchnorm_factor(built):
    x = np.ones((1, 2, 2, 3), np.float32)
    bn = {"gamma": np.ones(3), "beta": np.zeros(3), "mean": np.zeros(3), "var": np.ones(3)}
    y = oracle.batchnorm(x, bn)
    assert np.allclose(y, 1 / np.sqrt(1.001), rtol=1e-6)
    # variance clamp: sqrt(var + 1e-3) >= 1e-4 always; negative variance hits the clamp
    bn2 = {"gamma": np.ones(3), "beta": np.zeros(3), "mean": np.zeros(3), "var": np.full(3, -0.001)}
    assert np.allclose(oracle.batchnorm(x, bn2), 1 / 1e-4)


def test_depthwise_and_misc_known_answers(built):
    x = np.ones((1, 5, 5, 8), np.float32)
    w = np.arange(8 * 9, dtype=np.float32).reshape(8, 3, 3)
    y = oracle.depthwise(x, w, None, None, 1, 1, 1, "", 0, (5, 5))
    assert np.allclose(y[0, 2, 2], w.sum(axis=(1, 2)))
    assert np.allclose(y[0, 0, 0], w[:, 1:, 1:].sum(axis=(1, 2)))  # window clipped == zero padding
    # subpixel: component = x%r + r*(y%r), tanh always
    z = np.arange(1 * 2 * 2 * 4, dtype=np.float32).reshape(1, 2, 2, 4) / 10
    s = oracle.subpixel(z, 2)
    assert s.shape == (1, 4, 4, 1)
    assert np.isclose(s[0, 1, 0, 0], np.tanh(z[0, 0, 0, 2])) and np.isclose(s[0, 0, 1, 0], np.tanh(z[0, 0, 0, 1]))
    # nearest upsample, reflect pad, concat, argmax (1-based, first max)
    u = oracle.upsample(z, 2)
    assert np.array_equal(u[0, 2:4, 0:2], np.broadcast_to(z[0, 1, 0], (2, 2, 4)))
    p = oracle.pad(z, 1, 1, (4, 4), "reflect")
    assert np.array_equal(p[0, 0, 0], z[0, 1, 1])
    c = oracle.concat(z, 2 * z)
    assert np.array_equal(c[..., 4:], 2 * z)
    assert list(oracle.argmax1(np.array([[[[1, 5, 5, 2]]], [[[9, 0, 0, 0]]]], np.float32))) == [2, 1]
    # instance norm: mean 0, var 1 -> gamma, beta
    r = np.random.default_rng(0).standard_normal((2, 16, 16, 3)).astype(np.float32) * 3 + 1
    inn = oracle.instancenorm(r, np.ones(3), np.zeros(3))
    assert np.allclose(inn.mean(axis=(1, 2)), 0, atol=1e-5) and np.allclose(inn.var(axis=(1, 2)), 1, atol=1e-3)


def test_layout_roundtrip_c4hw4(built):
    r = np.random.default_rng(1).standard_normal((3, 5, 7)).astype(np.float32)  # H W C
    c4 = np.empty((2, 3, 5, 4), np.float32)
    oracle.lib().orc_hwc_to_c4hw4(r.ctypes.data_as(C.c_void_p), 3, 5, 7, c4.ctypes.data_as(C.c_void_p))
    assert c4[1, 2, 4, 2] == r[2, 4, 6] and c4[1, 0, 0, 3] == 0  # channels >= C are zero
    back = np.empty_like(r)
    oracle.lib().orc_c4hw4_to_hwc(c4.ctypes.data_as(C.c_void_p), 3, 5, 7, back.ctypes.data_as(C.c_void_p))
    assert np.array_equal(back, r)


def test_yolo_decode_known_answer(built):
    # one confident cell in head 0 (13x13 grid, anchor mask 3 -> 81x82), everything else far below threshold
    h0 = np.full((13, 13, 18), -10.0, np.float32)
    h1 = np.full((26, 26, 18), -10.0, np.float32)
    h0[6, 6, 0:6] = [0.0, 0.0, 0.0, 0.0, 10.0, 10.0]
    rows = oracle.yolo(h0, h1, (416, 416))
    assert rows.shape == (1, 6)
    cls, score, x, y, w, h = rows[0]
    assert cls == 0
    assert np.isclose(score, 1 / (1 + np.exp(-10.0) * (1 + np.exp(-10.0))), rtol=1e-6)  # yololayer.cpp:136 as parenthesised
    assert np.isclose(w, 81 / 416, rtol=1e-6) and np.isclose(h, 82 / 416, rtol=1e-6)
    assert np.isclose(x + w / 2, 6.5 / 13, rtol=1e-6)
    # a duplicate overlapping box is suppressed by NMS
    h0[6, 6, 6:12] = [0.0, 0.0, 0.0, 0.0, 9.0, 9.0]
    assert oracle.yolo(h0, h1, (416, 416)).shape[0] >= 1


def test_compare_is_the_reference_comparator(built):
    a = np.array([1.0, 100.0, 0.0, 1.0], np.float32)
    b = np.array([1.005, 100.5, 0.009, 1.02], np.float32)
    assert oracle.compare(a, b, 0.01) == 1  # |d|<=eps, rel<eps, |d|<=eps, fail
