"""GPU parity of the HEADLINE path: `frr_rpn_proposals` at BASELINE configs[1] (B = 64 images of 608x1008,
N = 21 546 anchors, 12 000 -> 2 000 @ IoU 0.7) and the bucketed NMS variant it selects, against the CPU oracle on
identical fp32 inputs (the GPU's own decoded boxes), image by image -- eager call and CUDA-graph replay.
Reference: RegionProposal.forward, models/model.py:44-55."""
import numpy as np
import pytest
import torch

import nms_cases
from faster_rcnn_pytorch_b200 import ops, region, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
HW = (608, 1008)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _inputs(B, seed0, hw=HW):
    ins = [synth.rpn_head_outputs(seed0 + i, hw) for i in range(B)]
    return np.stack([x[0] for x in ins]), np.stack([x[1] for x in ins]), np.stack([x[2] for x in ins])


def _check_plan_outputs(oracle, plan, rois, count, scores_in, pre_k, post_k, thr=0.7):
    """Every image: top-k order, keep list, count and rois bit-exact vs the oracle fed the GPU's decoded boxes."""
    it = {k: v.cpu().numpy() for k, v in plan.intermediates().items()}
    rois, count = rois.cpu().numpy(), count.cpu().numpy()
    B = rois.shape[0]
    for i in range(B):
        boxes, valid = it["boxes"][i], it["valid"][i].astype(bool)
        assert np.array_equal(valid, oracle.min_size_mask(boxes)), i
        sc = it["scores"][i] if scores_in is None else scores_in[i]
        src = np.nonzero(valid)[0]
        order = src[oracle.sort_desc(sc[valid])[:pre_k]]
        n = len(order)
        assert it["top_count"][i] == n, i
        assert np.array_equal(it["top_idx"][i, :n], order), i
        tb = boxes[order]
        want = oracle.nms(tb, -np.arange(n, dtype=np.float32), thr)[:post_k]
        c = int(count[i])
        assert c == len(want), (i, c, len(want))
        assert np.array_equal(it["keep"][i, :c], want), i
        assert (it["keep"][i, c:] == -1).all(), i
        assert np.array_equal(rois[i, :c], tb[want]), i
        assert not rois[i, c:].any(), i


def test_headline_config1_every_image_eager_and_graph(oracle):
    """configs[1] exactly: B = 64, 608x1008, 12000 -> 2000.  The variant the bench times must be the bucketed one."""
    B, n = 64, synth.num_anchors(HW)
    v = ops.nms_variant(B, 12000, 0.7, 2000, unit_boxes=True)
    assert v["variant"] == "bucketed", v
    lg, rg, sc = _inputs(B, 2000)
    plan = region.ProposalPlan(B, n, DEV, image_hw=HW, mode="train", logits=False)
    d_sc, d_rg = dev(sc), dev(rg)
    rois, count = plan.run(d_sc, d_rg)
    torch.cuda.synchronize()
    _check_plan_outputs(oracle, plan, rois.clone(), count.clone(), sc, 12000, 2000)
    assert int(count.min()) == 2000                       # the walk stops by max_keep on every image
    # CUDA-graph replay on NEW inputs in the captured buffers
    graph = plan.capture(d_sc, d_rg)
    lg2, rg2, sc2 = _inputs(B, 5000)
    d_sc.copy_(dev(sc2)); d_rg.copy_(dev(rg2))
    graph.replay()
    torch.cuda.synchronize()
    _check_plan_outputs(oracle, plan, plan.rois.clone(), plan.count.clone(), sc2, 12000, 2000)


def test_proposal_pipeline_batches_in_flight(oracle):
    """region.ProposalPipeline (the bench's throughput mode): four batches in flight on four streams, NMS with one CTA per
    image (frr_rpn_proposals with nms_cluster_size = 1), graph replays.  Every image of every batch against the oracle,
    and bit-equal to the single-plan / automatic-cluster result."""
    B, n = 64, synth.num_anchors(HW)
    v = ops.nms_variant(B, 12000, 0.7, 2000, cluster_size=1, unit_boxes=True)
    assert v["variant"] == "bucketed" and v["cluster_size"] == 1, v
    pipe = region.ProposalPipeline(B, n, DEV, depth=4, image_hw=HW, mode="train", logits=False)
    plan = region.ProposalPlan(B, n, DEV, image_hw=HW, mode="train", logits=False)
    batches = []
    for t in range(4):
        _, rg, sc = _inputs(B, 2000 + 100 * t)
        batches.append((sc, dev(sc), dev(rg)))
    for _, d_sc, d_rg in batches[:2]:
        pipe.capture(d_sc, d_rg)                          # two of the batches replay graphs, two run eagerly
    tickets = [pipe.submit(d_sc, d_rg) for _, d_sc, d_rg in batches]
    with pytest.raises(ValueError):
        pipe.result(tickets[-1] + 1)
    outs = []
    for t in tickets:
        rois, count = pipe.result(t)
        outs.append((rois.clone(), count.clone()))
    torch.cuda.synchronize()
    for t, (sc, d_sc, d_rg) in enumerate(batches):
        _check_plan_outputs(oracle, pipe.plans[t % 4], outs[t][0], outs[t][1], sc, 12000, 2000)
        r1, c1 = plan.run(d_sc, d_rg)
        assert torch.equal(r1, outs[t][0]) and torch.equal(c1, outs[t][1])
    # the buffers of a step are reused `depth` submits later
    pipe.submit(batches[0][1], batches[0][2])
    with pytest.raises(ValueError):
        pipe.result(tickets[0])
    pipe.drain()
    torch.cuda.synchronize()


def test_headline_logits_path_matches_scores_path_ordering(oracle):
    """Same call with [B,N,2] logits (what bench.py feeds): index-valued outputs checked on the GPU's own scores."""
    B, n = 64, synth.num_anchors(HW)
    rs = np.random.RandomState(2000)
    lg = rs.standard_normal((B, n, 2)).astype(np.float32)
    rg = (rs.standard_normal((B, n, 4)) * 0.2).astype(np.float32)
    plan = region.ProposalPlan(B, n, DEV, image_hw=HW, mode="train", logits=True)
    rois, count = plan.run(dev(lg), dev(rg))
    torch.cuda.synchronize()
    sc = plan.intermediates()["scores"].cpu().numpy()
    # softmax scores of N(0,1) logits collide now and then: the kernel's order is (score desc, index asc) = a stable
    # sort, which oracle.sort_desc reproduces (np stable argsort)
    _check_plan_outputs(oracle, plan, rois, count, None, 12000, 2000)
    np.testing.assert_allclose(sc[0], oracle.fg_softmax(lg[0]), rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("B", [19, 50, 75])
def test_plan_batch_sizes_that_pick_1_2_4_ctas_per_image(oracle, B):
    """auto cluster size 4 / 2 / 1 (148 SMs / B): all must take the bucketed variant and stay bit-exact."""
    hw = (320, 480)
    n = synth.num_anchors(hw)
    v = ops.nms_variant(B, min(12000, n), 0.7, 2000, unit_boxes=True)
    assert v["variant"] == "bucketed" and v["cluster_size"] == {19: 4, 50: 2, 75: 1}[B], v
    lg, rg, sc = _inputs(B, 300 + B, hw)
    plan = region.ProposalPlan(B, n, DEV, image_hw=hw, mode="train", logits=False)
    rois, count = plan.run(dev(sc), dev(rg))
    torch.cuda.synchronize()
    _check_plan_outputs(oracle, plan, rois, count, sc, 12000, 2000)


def _run_nms(b, thr, max_keep, **kw):
    keep, cnt, rois = ops.nms_sorted(dev(b[None]), thr, max_keep=max_keep, **kw)
    c = int(cnt[0])
    k = keep[0, :c].cpu().numpy()
    assert (keep[0, c:].cpu().numpy() == -1).all()
    assert np.array_equal(rois[0, :c].cpu().numpy(), b[k])
    return k


@pytest.mark.parametrize("thr", [0.7, 0.5, 0.3])
@pytest.mark.parametrize("name", nms_cases.ALL)
def test_bucketed_nms_adversarial_sets(oracle, name, thr):
    """Sets on the pruning boundaries (area-class edges, x-bin edges, IoU = thr at the extremal area ratio / centre
    distance, degenerate boxes, one class, piles of duplicates, sparse) through every geometry of the bucketed variant,
    against the oracle and against the un-bucketed kernel."""
    n = 6000
    b = nms_cases.make(name, 21, n, thr)
    n = len(b)
    for max_keep in (2000, 700):
        want = oracle.nms(b, -np.arange(n, dtype=np.float32), thr)[:max_keep]
        plain = _run_nms(b, thr, max_keep, cluster_size=8, threads=512)             # keep-list kernel, no buckets
        assert np.array_equal(plain, want), (name, thr, "plain")
        for cs, threads in [(1, 1024), (2, 1024), (4, 1024), (16, 1024), (1, 256), (2, 512), (8, 512), (16, 256)]:
            v = ops.nms_variant(1, n, thr, max_keep, cluster_size=cs, threads=threads, unit_boxes=True)
            assert v["variant"] == "bucketed" and v["cluster_size"] == cs and v["threads"] == threads, v
            got = _run_nms(b, thr, max_keep, cluster_size=cs, threads=threads, unit_boxes=True)
            assert np.array_equal(got, want), (name, thr, max_keep, cs, threads)


@pytest.mark.parametrize("cs", [1, 2, 4])
def test_bucketed_nms_batched_ragged_counts(oracle, cs):
    """Ragged batch through the bucketed variant: full, one short of a chunk, tiny, empty, single box."""
    B, n = 6, 5000
    bs = [nms_cases.rpn_like(700 + i, n, hw=(320, 480)) if i % 2 == 0 else nms_cases.make("dense_duplicates", 30 + i, n)
          for i in range(B)]
    n = min(len(x) for x in bs)
    bs = [x[:n] for x in bs]
    counts = np.array([n, n - 1, 2049, 257, 0, 1], np.int32)
    assert ops.nms_variant(B, n, 0.7, 2000, cluster_size=cs, unit_boxes=True)["variant"] == "bucketed"
    keep, cnt, rois = ops.nms_sorted(dev(np.stack(bs)), 0.7, max_keep=2000, counts=dev(counts), cluster_size=cs,
                                     unit_boxes=True)
    for i in range(B):
        c = counts[i]
        want = oracle.nms(bs[i][:c], -np.arange(c, dtype=np.float32), 0.7)[:2000]
        got = keep[i, :int(cnt[i])].cpu().numpy()
        assert np.array_equal(got, want), i
        assert np.array_equal(rois[i, :len(got)].cpu().numpy(), bs[i][got]), i


def test_bucketed_nms_walk_ends_by_count_with_a_partial_last_chunk(oracle):
    """max_keep never reached: every candidate is visited, the last chunk is partial."""
    for n in (2900, 1025, 255):
        b = nms_cases.rpn_like(2003, n)
        want = oracle.nms(b, -np.arange(len(b), dtype=np.float32), 0.7)
        assert len(want) < 2000
        for cs in (1, 2, 16):
            assert ops.nms_variant(1, len(b), 0.7, 2000, cluster_size=cs, unit_boxes=True)["variant"] == "bucketed"
            got = _run_nms(b, 0.7, 2000, cluster_size=cs, unit_boxes=True)
            assert np.array_equal(got, want), (n, cs)


@pytest.mark.parametrize("first,largest,lanes", [(256, 256, 1), (256, 2048, 32), (2048, 2048, 2), (512, 1024, 8)])
def test_bucketed_nms_result_does_not_depend_on_per_call_chunk_sizes(oracle, first, largest, lanes):
    tune = dict(first_chunk=first, max_chunk=largest, lanes_screen=lanes, lanes_pairs=lanes)
    for name in ("rpn_like", "dense_duplicates", "staircase"):
        b = nms_cases.make(name, 5, 7000)
        want = oracle.nms(b, -np.arange(len(b), dtype=np.float32), 0.7)[:2000]
        for cs in (1, 2, 8):
            got = _run_nms(b, 0.7, 2000, cluster_size=cs, unit_boxes=True, **tune)
            assert np.array_equal(got, want), (name, cs)
