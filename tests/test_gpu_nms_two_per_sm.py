"""The bucketed NMS with one CTA per image, in the automatic 1024-thread form and in the 512-thread form (chunks of at
most 1024 candidates) whose shared-memory layout fits twice per SM: bit for bit against the oracle and the keep-list
kernel, with neighbouring CTAs at very different phases, at the edge-region and hit-ring capacities of the smaller
layout, and with a chunk size request above its cap."""
import numpy as np
import pytest
import torch

import nms_cases
from faster_rcnn_pytorch_b200 import ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
HW = (608, 1008)
TWO_PER_SM_SMEM = 115712  # (228 KB per SM - 1 KB reserved per CTA) / 2


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _one_cta_forms(B, n, thr=0.7, max_keep=2000):
    v = ops.nms_variant(B, n, thr, max_keep, cluster_size=1, unit_boxes=True)
    assert v["variant"] == "bucketed" and v["cluster_size"] == 1 and v["threads"] == 1024, v
    v = ops.nms_variant(B, n, thr, max_keep, cluster_size=1, threads=512, unit_boxes=True)
    assert v["variant"] == "bucketed" and v["threads"] == 512 and v["smem"] <= TWO_PER_SM_SMEM, v
    return (0, 512)


def _keep_lists(keep, cnt):
    keep, cnt = keep.cpu().numpy(), cnt.cpu().numpy()
    for i in range(keep.shape[0]):
        assert (keep[i, cnt[i]:] == -1).all(), i
    return [keep[i, :cnt[i]] for i in range(keep.shape[0])]


def _check_batch(oracle, boxes, counts, thr=0.7, max_keep=2000):
    """Every image of both one-CTA-per-image forms against the keep-list kernel and the oracle."""
    B, n = boxes.shape[0], boxes.shape[1]
    d_b, d_c = dev(boxes), dev(counts)
    pk, pc, _ = ops.nms_sorted(d_b, thr, max_keep=max_keep, counts=d_c, cluster_size=8, threads=512)  # keep-list kernel
    plain = _keep_lists(pk, pc)
    want = []
    for i in range(B):
        c = int(counts[i])
        want.append(oracle.nms(boxes[i, :c], -np.arange(c, dtype=np.float32), thr)[:max_keep])
        assert np.array_equal(plain[i], want[i]), (i, "keep-list kernel")
    for threads in _one_cta_forms(B, n, thr, max_keep):
        keep, cnt, rois = ops.nms_sorted(d_b, thr, max_keep=max_keep, counts=d_c, cluster_size=1, threads=threads,
                                         unit_boxes=True)
        got = _keep_lists(keep, cnt)
        rois = rois.cpu().numpy()
        for i in range(B):
            assert np.array_equal(got[i], want[i]), (i, threads)
            assert np.array_equal(rois[i, :len(want[i])], boxes[i, want[i]]), (i, threads)


@pytest.mark.parametrize("thr", [0.7, 0.5])
def test_one_cta_forms_adversarial_and_boundary_sets(oracle, thr):
    sets = [nms_cases.make(name, 41, 6000, thr) for name in nms_cases.ALL]
    n = min(len(b) for b in sets)
    boxes = np.stack([b[:n] for b in sets])
    _check_batch(oracle, boxes, np.full(len(sets), n, np.int32), thr)


@pytest.mark.parametrize("B", [64, 19, 75])
def test_one_cta_forms_headline_batch(oracle, B):
    """The configs[1] shape (12 000 -> 2 000 at IoU 0.7) on decoded, top-k sorted RPN boxes."""
    ins = [synth.rpn_head_outputs(3000 + i, HW) for i in range(B)]
    reg = dev(np.stack([x[1] for x in ins]))
    sc = dev(np.stack([x[2] for x in ins]))
    boxes, scores, valid = ops.rpn_decode(reg, sc, image_hw=HW)
    top = ops.topk_desc(scores, 12000, valid=valid, boxes=boxes)
    _check_batch(oracle, top["boxes"].cpu().numpy(), top["count"].cpu().numpy())


def test_neighbouring_ctas_with_very_different_work(oracle):
    """Counts of 0, 1, 300 and 12 000, images alternating between piles of near-duplicates and spread-out boxes: two
    CTAs that share an SM are at very different phases of their walks."""
    B, n = 24, 12000
    boxes = np.stack([nms_cases.dense_duplicates(60 + i, n) if i % 2 == 0 else nms_cases.sparse(60 + i, n)
                      for i in range(B)])
    counts = np.array([(0, 1, 300, 12000)[(i // 2) % 4] for i in range(B)], np.int32)
    _check_batch(oracle, boxes, counts)


def _identical_boxes(seed, sites, per_site, n):
    """`sites` piles of `per_site` identical boxes (decreasing scores), then small, hardly overlapping boxes up to n
    (they add next to no edges of their own)."""
    rs = np.random.RandomState(seed)
    c = rs.uniform(0.2, 0.8, (sites, 2))
    wh = rs.uniform(0.05, 0.2, (sites, 2))
    pile = np.concatenate([c - wh / 2, c + wh / 2], axis=1).astype(np.float32)
    head = np.repeat(pile, per_site, axis=0)
    return np.concatenate([head, nms_cases.sparse(seed, n - len(head))]).astype(np.float32)


@pytest.mark.parametrize("sites,per_site", [(1, 600), (2, 400), (3, 24)])
def test_edge_region_and_hit_ring_overflow(oracle, sites, per_site):
    """One pile of 600 (or two of 400) identical boxes in the first chunk gives ~180 k suppression pairs, far more
    than the 2048 edges of the region; three piles of 24 stay inside the region but overflow the 4-entry hit ring
    of every lane that walks a pile."""
    n = 4000
    b = _identical_boxes(70 + sites, sites, per_site, n)
    _check_batch(oracle, b[None], np.array([n], np.int32))


def test_chunk_request_above_the_cap_is_clamped(oracle):
    """The 512-thread form holds chunks of 1024 candidates: a request for 2048 runs with 1024."""
    b = nms_cases.rpn_like(2024, 9000)
    n = len(b)
    d_b = dev(b[None])
    want = oracle.nms(b, -np.arange(n, dtype=np.float32), 0.7)[:2000]
    auto, ac, _ = ops.nms_sorted(d_b, 0.7, max_keep=2000, cluster_size=1, unit_boxes=True)
    assert np.array_equal(_keep_lists(auto, ac)[0], want)
    for first in (0, 2048):
        keep, cnt, _ = ops.nms_sorted(d_b, 0.7, max_keep=2000, cluster_size=1, threads=512, unit_boxes=True,
                                      first_chunk=first, max_chunk=2048)
        assert np.array_equal(_keep_lists(keep, cnt)[0], want), first
