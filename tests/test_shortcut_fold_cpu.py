"""CPU tests of the folded projection shortcut's K walk (csrc/kernels_umma.cu: decode_kblock / for_each_kblock, fed with the work items of
decode_work and of the stream-K schedule), evaluated on the host through snnb_debug_kblock_schedule: every K block of the concatenated K
[k*k taps x cblocks | shortcut cblocks] of every tile is loaded exactly once, from the right operand, tap and channel block, at the right
weight column - also when a split-K or stream-K range straddles the end of the taps."""
import ctypes as C

import numpy as np
import pytest

from shadernn_b200._lib import lib


def walk(ksize, cblocks, icp, sc_cblocks, tiles, ksplit, sms=148):
    num_kb = ksize * ksize * cblocks + sc_cblocks
    cap = tiles * num_kb + 16
    rows = np.zeros((cap, 6), np.int32)
    n = lib().snnb_debug_kblock_schedule(ksize, cblocks, icp, sc_cblocks, tiles, ksplit, sms, rows.ctypes.data_as(C.POINTER(C.c_int)), cap)
    assert n <= cap
    return None if n < 0 else rows[:n]


def expected(kb, ksize, cblocks, icp):
    """(shortcut, tap, channel block, weight column) of K block kb: taps first, tap-major; then the shortcut's blocks."""
    kb_main = ksize * ksize * cblocks
    if kb < kb_main:
        tap, cb = divmod(kb, cblocks)
        return 0, tap, cb, tap * icp + cb * 64
    return 1, 0, kb - kb_main, ksize * ksize * icp + (kb - kb_main) * 64


# ResNet-18's down-sampling blocks (k 3, IC = OC, shortcut IC = OC / 2) and odd channel counts (IC 40 -> pitch 40, shortcut 24)
SHAPES = [
    (3, 2, 128, 1, 224),   # 28x28x128: 18 + 1 K blocks
    (3, 4, 256, 2, 128),   # 14x14x256: 36 + 2
    (3, 8, 512, 4, 52),    # 7x7x512:   72 + 4 (the split-K layer)
    (3, 1, 40, 1, 7),      # IC 40, shortcut 24: both one partial channel block
    (1, 2, 128, 3, 300),   # a 1x1 convolution (bottleneck expansion) with a wider shortcut
    (3, 2, 128, 0, 10),    # no shortcut: the walk is the plain tap loop
]


@pytest.mark.parametrize("ksize,cblocks,icp,sc_cblocks,tiles", SHAPES)
@pytest.mark.parametrize("ksplit", [1, 2, 3, 0])  # 0 = stream-K
def test_every_k_block_once_with_its_operand_and_weight_column(ksize, cblocks, icp, sc_cblocks, tiles, ksplit):
    num_kb = ksize * ksize * cblocks + sc_cblocks
    rows = walk(ksize, cblocks, icp, sc_cblocks, tiles, ksplit)
    if rows is None:
        assert ksplit == 0  # stream-K declines when there is nothing to cut
        return
    cover = np.zeros((tiles, num_kb), np.int32)
    for tile, kb, sc, tap, cb, wcol in rows.tolist():
        assert 0 <= tile < tiles and 0 <= kb < num_kb
        cover[tile, kb] += 1
        assert (sc, tap, cb, wcol) == expected(kb, ksize, cblocks, icp), (kb, sc, tap, cb, wcol)
    assert (cover == 1).all(), "K blocks loaded %s times" % sorted(set(cover.ravel().tolist()))


@pytest.mark.parametrize("ksplit", [2, 3])
def test_split_ranges_straddle_the_shortcut(ksplit):
    # 7x7x512: 72 + 4 K blocks. ksplit 2: ranges [0, 38) [38, 76); ksplit 3: [0, 26) [26, 52) [52, 76) - the last range of every tile runs
    # from the taps into the shortcut. Each work item's rows are one consecutive K range, and the operand switches at most once.
    rows = walk(3, 8, 512, 4, 4, ksplit)
    runs = []
    for r in rows.tolist():
        if runs and runs[-1][-1][0] == r[0] and runs[-1][-1][1] + 1 == r[1]:
            runs[-1].append(r)
        else:
            runs.append([r])
    straddles = 0
    for run in runs:
        sc = [r[2] for r in run]
        assert sc == sorted(sc)  # taps, then shortcut: never back
        straddles += 0 < sum(sc) < len(sc)
    assert straddles == 4


def test_stream_k_pieces_straddle_the_shortcut():
    # 28x28x128 folded: 224 tiles of 19 K blocks on 148 SMs -> 76 tiles cut into pieces; a tile's pieces still cover it once, in K order
    # up to the shortcut block 18
    rows = walk(3, 2, 128, 1, 224, 0)
    by_tile = {}
    for tile, kb, sc, *_ in rows.tolist():
        by_tile.setdefault(tile, []).append((kb, sc))
    assert all(sorted(kb for kb, _ in v) == list(range(19)) for v in by_tile.values())
    assert all(sc == (kb == 18) for v in by_tile.values() for kb, sc in v)


def test_invalid_arguments_are_refused():
    assert lib().snnb_debug_kblock_schedule(0, 1, 64, 0, 1, 1, 148, None, 0) == -1
    assert lib().snnb_debug_kblock_schedule(3, 1, 64, -1, 1, 1, 148, None, 0) == -1
    assert lib().snnb_debug_kblock_schedule(3, 2, 128, 1, 296, 0, 148, None, 0) == -1  # stream-K: whole waves only, nothing to cut
