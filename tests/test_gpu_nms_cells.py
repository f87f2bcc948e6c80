"""The bucketed NMS with (x bin, y bin, area class) keys, in every launch form -- one CTA per image, clusters of 2 and 4
per image, and the forms that key by x bin only: single-image clusters of 8 and 16 and the 512-thread form -- bit for
bit against the oracle on the sets of nms_cases.py with x and y swapped (the x-bin-edge and x-cut-extremal sets then
sit on the y cell edges and the y cut) and on boxes whose centres lie exactly on cell edges."""
import numpy as np
import pytest
import torch

import nms_cases
from faster_rcnn_pytorch_b200 import ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MAX_KEEP = 2000
# (cluster_size, threads, images per launch)
FORMS = [(1, 0, None), (2, 0, None), (4, 0, None), (8, 0, 1), (16, 0, 1), (1, 512, None)]


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def mirrored(b):
    return np.ascontiguousarray(b[:, [1, 0, 3, 2]])


def cell_edges(seed: int, n: int):
    """x- and y-centres exactly on the cell edges j/8 (the y edges j/4 among them; dyadic widths and heights: the fp32
    centre is exact), a third of them nudged one ulp across the edge in x, y or both, with copies that overlap across
    the edge."""
    rs = np.random.RandomState(seed)
    c = rs.randint(0, 9, (n, 2)) / 8.0
    wh = 2.0 ** -rs.randint(2, 9, (n, 2)).astype(np.float64)
    b = np.concatenate([c - wh / 2, c + wh / 2], axis=1).astype(np.float32)
    k = rs.randint(0, 4, n)
    for ax, sel in ((0, (k == 1) | (k == 3)), (1, (k == 2) | (k == 3))):
        d = np.where(rs.randint(0, 2, n) == 0, np.float32(-1.0), np.float32(2.0))
        b[sel, ax] = np.nextafter(b[sel, ax], d[sel])
        b[sel, ax + 2] = np.nextafter(b[sel, ax + 2], d[sel])
    j = rs.randint(0, n, n // 3)
    b[j] += np.float32(1e-4)
    return np.clip(b, 0.0, 1.0).astype(np.float32)


def _check(oracle, sets, thr):
    n = min(len(b) for b in sets)
    boxes = np.stack([b[:n] for b in sets])
    counts = np.full(len(sets), n, np.int32)
    want = [oracle.nms(b, -np.arange(n, dtype=np.float32), thr)[:MAX_KEEP] for b in boxes]
    for S, threads, per_launch in FORMS:
        step = per_launch or len(sets)
        for i0 in range(0, len(sets), step):
            B = min(step, len(sets) - i0)
            v = ops.nms_variant(B, n, thr, MAX_KEEP, cluster_size=S, threads=threads, unit_boxes=True)
            assert v["variant"] == "bucketed" and v["cluster_size"] == S, v
            keep, cnt, rois = ops.nms_sorted(dev(boxes[i0:i0 + B]), thr, max_keep=MAX_KEEP, counts=dev(counts[i0:i0 + B]),
                                             cluster_size=S, threads=threads, unit_boxes=True)
            keep, cnt, rois = keep.cpu().numpy(), cnt.cpu().numpy(), rois.cpu().numpy()
            for b in range(B):
                w = want[i0 + b]
                form = (S, threads, i0 + b)
                assert cnt[b] == len(w), form
                assert np.array_equal(keep[b, :cnt[b]], w), form
                assert (keep[b, cnt[b]:] == -1).all(), form
                assert np.array_equal(rois[b, :cnt[b]], boxes[i0 + b, w]), form
                assert not rois[b, cnt[b]:].any(), form


@pytest.mark.parametrize("thr", [0.7, 0.5])
def test_mirrored_sets_every_form(oracle, thr):
    _check(oracle, [mirrored(nms_cases.make(name, 43, 6000, thr)) for name in nms_cases.ALL], thr)


@pytest.mark.parametrize("thr", [0.7, 0.5, 0.3])
def test_cell_edge_boxes_every_form(oracle, thr):
    _check(oracle, [cell_edges(90 + i, 5000) for i in range(4)], thr)
