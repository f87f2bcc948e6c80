"""CPU: the walks of the bucketed NMS kernel over (x bin, y bin, area class) keys (tests/nms_cell_model.py) keep exactly
what the oracle (= torchvision's CPU kernel) keeps, visit every pair that can suppress, and meet each pair among a
chunk's survivors exactly once, from its lower bucketed position -- on every set of nms_cases.py and on its copy with
x and y swapped, which puts the x-bin-edge and x-cut-extremal sets on the y cell edges and the y cut."""
import numpy as np
import pytest

import nms_cases
import nms_cell_model


def mirrored(b):
    return np.ascontiguousarray(b[:, [1, 0, 3, 2]])


@pytest.mark.parametrize("mirror", [False, True], ids=["xy", "yx"])
@pytest.mark.parametrize("thr", [0.7, 0.5, 0.3])
@pytest.mark.parametrize("name", nms_cases.ALL)
def test_cell_walks_equal_oracle(oracle, name, thr, mirror):
    b = nms_cases.make(name, 11, 3000, thr)
    if mirror:
        b = mirrored(b)
    want = oracle.nms(b, -np.arange(len(b), dtype=np.float32), thr)[:1000]
    for chunks in [(2048,), (512, 1024, 256)]:
        st = {}
        got = nms_cell_model.nms_cells(b, thr, 1000, chunk_sizes=chunks, stats=st)
        assert np.array_equal(got, want), (name, thr, chunks)
        assert st["missed_d"] == 0 and st["missed_h"] == 0, st
        assert st["twice_h"] == 0 and st["down_h"] == 0, st


def test_x_only_key_of_the_smaller_layouts():
    """ky = 1 (the 256/512-thread layouts and the large clusters) keeps what ky = 4 keeps, and tests more pairs."""
    b = nms_cases.make("x_bin_edges", 12, 3000, 0.7)
    st1, st4 = {}, {}
    k1 = nms_cell_model.nms_cells(b, 0.7, 1000, ky=1, stats=st1)
    k4 = nms_cell_model.nms_cells(b, 0.7, 1000, ky=4, stats=st4)
    assert np.array_equal(k1, k4)
    assert st1["missed_d"] == st1["missed_h"] == st1["twice_h"] == st1["down_h"] == 0
    assert st4["pairs_d"] + st4["pairs_h"] < st1["pairs_d"] + st1["pairs_h"]


def test_cells_cut_rpn_pair_tests():
    """On RPN proposals the y cut of the 1024-thread grid removes half of the pairs the x-only key tests; the keep
    list is unchanged."""
    b = nms_cases.rpn_like(2000, 12000)
    st1, st4 = {}, {}
    k1 = nms_cell_model.nms_cells(b, 0.7, 2000, chunk_sizes=(1024, 2048), ky=1, stats=st1)
    k4 = nms_cell_model.nms_cells(b, 0.7, 2000, chunk_sizes=(1024, 2048), ky=4, stats=st4)
    assert np.array_equal(k1, k4)
    assert st4["missed_d"] == st4["missed_h"] == st4["twice_h"] == 0
    assert 2 * (st4["pairs_d"] + st4["pairs_h"]) < st1["pairs_d"] + st1["pairs_h"], (st1, st4)
