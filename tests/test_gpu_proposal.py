"""GPU parity: CUDA proposal path (decode -> top-k -> NMS) vs the CPU oracle, through the C ABI.
Bit-exact for index-valued outputs from identical fp32 inputs; 1e-5 relative for exp()-bearing floats."""
import numpy as np
import pytest
import torch

from conftest import golden, sha
from faster_rcnn_pytorch_b200 import ops, synth

pytestmark = pytest.mark.gpu
RTOL = 1e-5
DEV = "cuda:0"


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


# ------------------------------------------------------------------------------------ anchors
@pytest.mark.parametrize("hw", [(64, 96), (600, 1000), (608, 1008), (800, 1333), (800, 800), (16, 16)])
def test_anchors_bit_exact(oracle, hw):
    a = ops.anchors(hw, DEV).cpu().numpy()
    assert np.array_equal(a, oracle.enumerate_anchors(hw))
    g = golden("anchors")
    key = f"{hw[0]}x{hw[1]}"
    if f"sha_{key}" in g:
        assert np.array_equal(sha(a), g[f"sha_{key}"])


# ------------------------------------------------------------------------------------ decode
@pytest.mark.parametrize("hw,seed,B", [((160, 256), 200, 1), ((600, 1000), 1000, 2), ((608, 1008), 2000, 3), ((800, 1333), 4000, 1)])
@pytest.mark.parametrize("gen_anchors", [True, False])
def test_rpn_decode_matches_oracle(oracle, hw, seed, B, gen_anchors):
    ins = [synth.rpn_head_outputs(seed + i, hw) for i in range(B)]
    logits = np.stack([x[0] for x in ins]); reg = np.stack([x[1] for x in ins])
    anchor = oracle.enumerate_anchors(hw)
    if gen_anchors:
        boxes, scores, valid = ops.rpn_decode(dev(reg), dev(logits), image_hw=hw)
    else:
        boxes, scores, valid = ops.rpn_decode(dev(reg), dev(logits), anchors=dev(anchor))
    boxes, scores, valid = boxes.cpu().numpy(), scores.cpu().numpy(), valid.cpu().numpy().astype(bool)
    for i in range(B):
        np.testing.assert_allclose(scores[i], oracle.fg_softmax(logits[i]), rtol=RTOL, atol=1e-7)
        np.testing.assert_allclose(boxes[i], oracle.decode_clip(reg[i], anchor), rtol=RTOL, atol=1e-6)
        # the min-size test is an fp32 compare: bit-exact on the boxes the GPU produced
        assert np.array_equal(valid[i], oracle.min_size_mask(boxes[i]))
        assert valid[i].sum() < valid[i].size  # the filter is exercised


def test_rpn_decode_small_golden_and_scores_passthrough(oracle):
    g = golden("proposal")
    hw = (160, 256)
    logits, reg, scores = synth.rpn_head_outputs(200, hw)
    b, s, v = ops.rpn_decode(dev(reg[None]), dev(logits[None]), image_hw=hw)
    np.testing.assert_allclose(b[0].cpu().numpy(), g["small_train_boxes"], rtol=RTOL, atol=1e-6)
    np.testing.assert_allclose(s[0].cpu().numpy(), g["small_train_score"], rtol=RTOL, atol=1e-7)
    b2, s2, v2 = ops.rpn_decode(dev(reg[None]), dev(scores[None]), image_hw=hw)
    assert np.array_equal(s2[0].cpu().numpy(), scores) and torch.equal(b, b2) and torch.equal(v, v2)


def test_rpn_decode_rejects_cpu_and_bad_shapes():
    with pytest.raises(ValueError):
        ops.rpn_decode(torch.zeros(1, 9, 4), torch.zeros(1, 9, 2), image_hw=(16, 16))
    with pytest.raises(ValueError):
        ops.rpn_decode(torch.zeros(1, 10, 4, device=DEV), torch.zeros(1, 10, 2, device=DEV), image_hw=(16, 16))


# ------------------------------------------------------------------------------------ top-k
def _oracle_topk(oracle, scores, valid, k):
    src = np.nonzero(valid)[0]
    order = oracle.sort_desc(scores[valid])[:k]
    return order, src[order]


@pytest.mark.parametrize("N,k,seed", [(21546, 12000, 1), (20646, 6000, 2), (37350, 6000, 3), (37350, 12000, 4),
                                      (1440, 12000, 5), (100, 7, 6), (33, 33, 7), (5000, 1, 8)])
def test_topk_indices_bit_exact(oracle, N, k, seed):
    rs = np.random.RandomState(seed)
    B = 3
    scores = np.stack([synth.unique_scores(rs, N) for _ in range(B)])
    valid = rs.uniform(size=(B, N)) > 0.02
    boxes = rs.uniform(size=(B, N, 4)).astype(np.float32)
    r = ops.topk_desc(dev(scores), k, valid=dev(valid.astype(np.uint8)), boxes=dev(boxes), want_cidx=True)
    cnt = r["count"].cpu().numpy()
    for b in range(B):
        cidx, idx = _oracle_topk(oracle, scores[b], valid[b], k)
        n = len(idx)
        assert cnt[b] == n == min(k, valid[b].sum())
        assert np.array_equal(r["idx"][b, :n].cpu().numpy(), idx)
        assert np.array_equal(r["cidx"][b, :n].cpu().numpy(), cidx)
        assert np.array_equal(r["scores"][b, :n].cpu().numpy(), scores[b][idx])
        assert np.array_equal(r["boxes"][b, :n].cpu().numpy(), boxes[b][idx])
        assert (r["idx"][b, n:].cpu().numpy() == -1).all()
        assert np.isneginf(r["scores"][b, n:].cpu().numpy()).all()


def test_topk_ties_lower_index_first_and_no_valid_mask(oracle):
    rs = np.random.RandomState(9)
    N, k = 4000, 1500
    scores = (np.round(rs.uniform(size=(2, N)) * 50) / 50).astype(np.float32)   # ~80 duplicates per value
    scores[1, ::3] = -scores[1, ::3]                                           # negative keys and -0.0
    r = ops.topk_desc(dev(scores), k)
    for b in range(2):
        want = oracle.sort_desc(scores[b])[:k]
        # -0.0 and +0.0 compare equal on the CPU; the kernel orders -0 < +0: compare via (score, idx) where defined
        got = r["idx"][b].cpu().numpy()
        assert np.array_equal(scores[b][got], scores[b][want])
        nz = scores[b][want] != 0
        assert np.array_equal(got[nz], want[nz])
    assert r["cidx"] is None and (r["count"].cpu().numpy() == k).all()


def test_topk_golden_reference_indices(oracle):
    """top-k indices of the reference's own sort (tests/golden/topk_nms.npz), identical fp32 scores."""
    g = golden("topk_nms")
    for name, hw, seed, k in [("rpn_train", (608, 1008), 2000, 12000), ("voc_test", (600, 1000), 1000, 6000),
                              ("coco_test", (800, 1333), 4000, 6000), ("small", (160, 256), 200, 12000)]:
        _, reg, scores = synth.rpn_head_outputs(seed, hw)
        boxes = oracle.decode_clip(reg, oracle.enumerate_anchors(hw))     # CPU-decoded: same validity as the golden run
        valid = oracle.min_size_mask(boxes)
        r = ops.topk_desc(dev(scores[None]), k, valid=dev(valid[None].astype(np.uint8)), want_cidx=True)
        n = int(r["count"][0])
        assert np.array_equal(r["cidx"][0, :n].cpu().numpy(), g[f"{name}_topk_idx"])


# ------------------------------------------------------------------------------------ NMS
def _sorted_boxes(seed, n):
    b, s = synth.random_boxes(seed, n)
    o = np.argsort(-s.astype(np.float64), kind="stable")
    return b[o], s[o], o


def test_nms_kats(oracle):
    f = np.float32
    def run(b, thr):
        keep, cnt, _ = ops.nms_sorted(dev(np.asarray(b, f)[None]), thr)
        return keep[0, :int(cnt[0])].cpu().tolist()
    assert run([[0, 0, 5, 1], [2, 0, 10, 1]], 0.3) == [0]            # IoU == 0.3f > 0.3 (double compare)
    assert run([[0, 0, 7, 1], [0, 0, 10, 1]], 0.7) == [0, 1]         # 0.7f < 0.7
    assert run([[0, 0, 1, 1], [2, 2, 3, 3], [4, 4, 5, 5]], 0.5) == [0, 1, 2]
    assert run([[1, 1, 1, 1], [1, 1, 1, 1]], 0.5) == [0, 1]          # 0/0 = NaN never suppresses
    keep, cnt, rois = ops.nms_sorted(torch.zeros((1, 0, 4), device=DEV), 0.5, max_keep=5)
    assert int(cnt[0]) == 0 and (keep.cpu().numpy() == -1).all()


@pytest.mark.parametrize("key", ["rand_100_64_0.5", "rand_101_65_0.7", "rand_102_1000_0.7", "rand_103_3000_0.3",
                                 "rand_104_12000_0.7", "rand_105_6000_0.7", "rand_106_300_0.3", "rand_107_1_0.7",
                                 "rand_108_2500_0.0", "rand_109_2500_1.0"])
@pytest.mark.parametrize("cluster", [0, 1, 2, 16])
def test_nms_golden_torchvision_keep_lists(oracle, key, cluster):
    g = golden("nms")
    _, seed, n, thr = key.split("_")
    b, s, o = _sorted_boxes(int(seed), int(n))
    if int(n) > 8000 and cluster == 1:
        pytest.skip("kept list of a full 12000-box NMS needs >= 2 CTAs of shared memory (auto-grown elsewhere)")
    keep, cnt, rois = ops.nms_sorted(dev(b[None]), float(thr), cluster_size=cluster)
    k = keep[0, :int(cnt[0])].cpu().numpy()
    want = g[key].astype(np.int64)                    # indices into the unsorted input
    assert np.array_equal(o[k], want)
    assert np.array_equal(rois[0, :len(k)].cpu().numpy(), b[k])
    assert (keep[0, len(k):].cpu().numpy() == -1).all()


@pytest.mark.parametrize("cluster", [0, 1, 2, 4, 8, 16])
def test_nms_batched_max_keep_and_counts(oracle, cluster):
    B, n = 5, 3000
    bs = [_sorted_boxes(300 + i, n)[0] for i in range(B)]
    counts = np.array([3000, 2999, 257, 0, 1], np.int32)
    keep, cnt, rois = ops.nms_sorted(dev(np.stack(bs)), 0.7, max_keep=300, counts=dev(counts), cluster_size=cluster)
    for i in range(B):
        c = counts[i]
        want = oracle.nms(bs[i][:c], -np.arange(c, dtype=np.float32), 0.7)[:300]
        got = keep[i, :int(cnt[i])].cpu().numpy()
        assert np.array_equal(got, want)
        assert np.array_equal(rois[i, :len(got)].cpu().numpy(), bs[i][got])


def test_nms_degenerate_and_threshold_variants(oracle):
    rs = np.random.RandomState(5)
    b, _, _ = _sorted_boxes(400, 1500)
    b[::7, 2] = b[::7, 0]                 # zero width
    b[::11, [0, 2]] = b[::11, [2, 0]]     # x2 < x1 (malformed)
    b[5] = b[4]                            # exact duplicate
    for thr in (0.7, 0.5, 0.3, 1e-9, 0.0, -0.5, 1.0, 2.0, 0.699999988079071, float(np.float32(0.7))):
        keep, cnt, _ = ops.nms_sorted(dev(b[None]), thr)
        want = oracle.nms(b, -np.arange(len(b), dtype=np.float32), thr)
        assert np.array_equal(keep[0, :int(cnt[0])].cpu().numpy(), want), thr


def test_nms_exact_threshold_boundary_pairs(oracle):
    """Pairs engineered to sit on / next to the decision boundary exercise the guard band + exact path."""
    rs = np.random.RandomState(6)
    n = 2048
    w = rs.uniform(0.05, 0.3, n).astype(np.float32)
    b = np.zeros((n, 4), np.float32)
    b[:, 2] = w
    b[:, 3] = 0.1
    # box j+1 overlaps box j along x with IoU close to 0.7 or 0.3
    for j in range(0, n - 1, 2):
        t = 0.7 if (j // 2) % 2 == 0 else 0.3
        frac = np.float32(2 * t / (1 + t))           # equal-size boxes: IoU = f/(2-f)
        b[j + 1, 0] = b[j, 0] + b[j, 2] * (1 - frac)
        b[j + 1, 2] = b[j + 1, 0] + (b[j, 2] - b[j, 0])
        off = np.float32(j) * np.float32(0.5)
        b[j:j + 2, [0, 2]] += off                     # separate the pairs
    for thr in (0.7, 0.3):
        keep, cnt, _ = ops.nms_sorted(dev(b[None]), thr)
        want = oracle.nms(b, -np.arange(n, dtype=np.float32), thr)
        assert np.array_equal(keep[0, :int(cnt[0])].cpu().numpy(), want)


@pytest.mark.parametrize("name,hw,seed,pre_k,post_k", [("rpn_train", (608, 1008), 2000, 12000, 2000),
                                                       ("voc_test", (600, 1000), 1000, 6000, 300),
                                                       ("coco_test", (800, 1333), 4000, 6000, 300),
                                                       ("small", (160, 256), 200, 12000, 2000)])
def test_proposal_chain_against_reference_goldens(oracle, name, hw, seed, pre_k, post_k):
    """CPU-decoded boxes (bit-identical to the reference's) -> GPU top-k -> GPU NMS == reference keep list."""
    g = golden("topk_nms")
    _, reg, scores = synth.rpn_head_outputs(seed, hw)
    boxes = oracle.decode_clip(reg, oracle.enumerate_anchors(hw))
    valid = oracle.min_size_mask(boxes)
    r = ops.topk_desc(dev(scores[None]), pre_k, valid=dev(valid[None].astype(np.uint8)), boxes=dev(boxes[None]), want_cidx=True)
    keep, cnt, rois = ops.nms_sorted(r["boxes"], 0.7, max_keep=post_k, counts=r["count"])
    k = keep[0, :int(cnt[0])].cpu().numpy()
    assert np.array_equal(k, g[f"{name}_keep"])
    if np.array_equal(sha(boxes), g[f"{name}_boxes_sha"]):
        assert np.array_equal(sha(rois[0, :len(k)].cpu().numpy()), g[f"{name}_rois_sha"])


@pytest.mark.parametrize("hw,seed,mode,B", [((608, 1008), 2000, "train", 4), ((800, 1333), 4000, "test", 2)])
def test_full_gpu_proposal_pipeline_stagewise(oracle, hw, seed, mode, B):
    """logits/reg -> GPU decode -> GPU top-k -> GPU NMS; each stage checked against the oracle run on the
    previous GPU stage's output (identical fp32 inputs on both sides)."""
    pre_k, post_k = oracle.PROPOSAL_MODES[mode]
    ins = [synth.rpn_head_outputs(seed + i, hw) for i in range(B)]
    reg = np.stack([x[1] for x in ins]); scores = np.stack([x[2] for x in ins])
    boxes, sc, valid = ops.rpn_decode(dev(reg), dev(scores), image_hw=hw)
    r = ops.topk_desc(sc, pre_k, valid=valid, boxes=boxes, want_cidx=True)
    keep, cnt, rois = ops.nms_sorted(r["boxes"], 0.7, max_keep=post_k, counts=r["count"])
    bx, va = boxes.cpu().numpy(), valid.cpu().numpy().astype(bool)
    for i in range(B):
        n = int(r["count"][i])
        cidx, idx = _oracle_topk(oracle, scores[i], va[i], pre_k)
        assert np.array_equal(r["idx"][i, :n].cpu().numpy(), idx)
        tb = bx[i][idx]
        want = oracle.nms(tb, -np.arange(n, dtype=np.float32), 0.7)[:post_k]
        got = keep[i, :int(cnt[i])].cpu().numpy()
        assert np.array_equal(got, want)
        assert np.array_equal(rois[i, :len(got)].cpu().numpy(), tb[got])


# ------------------------------------------------------------------------------------ fused call / host pipeline
def test_proposal_plan_and_host_pipeline_match_stagewise_ops(oracle):
    """frr_rpn_proposals (one C-ABI call, caller workspace) and the double-buffered host pipeline return
    exactly what the three separate ops return."""
    from faster_rcnn_pytorch_b200 import region
    hw, B = (320, 480), 3
    ins = [synth.rpn_head_outputs(900 + i, hw) for i in range(2 * B)]
    n = synth.num_anchors(hw)
    for mode in ("train", "test"):
        plan = region.ProposalPlan(B, n, DEV, image_hw=hw, mode=mode, logits=True)
        pipe = region.HostProposalPipeline(plan)
        tickets, wants = [], []
        for s in range(2):
            lg = np.stack([x[0] for x in ins[s * B:(s + 1) * B]]); rg = np.stack([x[1] for x in ins[s * B:(s + 1) * B]])
            want_rois, want_cnt = region.rpn_proposals(dev(lg), dev(rg), image_hw=hw, mode=mode)
            rois, cnt = plan.run(dev(lg), dev(rg))
            assert torch.equal(rois, want_rois) and torch.equal(cnt, want_cnt)
            tickets.append(pipe.submit(lg, rg))
            wants.append((want_rois.cpu(), want_cnt.cpu()))
        for t, (wr, wc) in zip(tickets, wants):
            hr, hc = pipe.result(t)
            assert torch.equal(hr, wr) and torch.equal(hc, wc)
    with pytest.raises(ValueError):
        plan.run(torch.zeros(B, n, 2), torch.zeros(B, n, 4))


def test_nms_unit_range_screen_gives_identical_keep_lists(oracle):
    """unit_boxes=True (coordinates in [0,1]: cheaper screening test) must not change any result."""
    for seed, n, thr in [(104, 12000, 0.7), (103, 3000, 0.3), (400, 1500, 0.5)]:
        b, _, _ = _sorted_boxes(seed, n)
        if seed == 400:
            b[::7, 2] = b[::7, 0]; b[::11, [0, 2]] = b[::11, [2, 0]]; b[5] = b[4]
        k0, c0, r0 = ops.nms_sorted(dev(b[None]), thr, max_keep=2000)
        k1, c1, r1 = ops.nms_sorted(dev(b[None]), thr, max_keep=2000, unit_boxes=True)
        assert torch.equal(k0, k1) and torch.equal(c0, c1) and torch.equal(r0, r1)
        want = oracle.nms(b, -np.arange(n, dtype=np.float32), thr)[:2000]
        assert np.array_equal(k1[0, :int(c1[0])].cpu().numpy(), want)


def test_nms_indirect_order_matches_gathered_boxes(oracle):
    """frr_nms_sorted_indirect(boxes_src, order) == frr_nms_sorted(boxes_src[order])."""
    from faster_rcnn_pytorch_b200 import _lib
    lib = _lib.load()
    B, N, k = 3, 5000, 3000
    rs = np.random.RandomState(77)
    src = np.stack([synth.random_boxes(600 + i, N)[0] for i in range(B)])
    order = np.stack([rs.permutation(N)[:k] for _ in range(B)]).astype(np.int32)
    counts = np.asarray([k, k - 7, 100], np.int32)
    gathered = np.stack([src[i][order[i]] for i in range(B)])
    want_keep, want_cnt, want_rois = ops.nms_sorted(dev(gathered), 0.7, max_keep=500, counts=dev(counts))
    d_src, d_ord, d_cnt = dev(src), dev(order), dev(counts)
    keep = torch.empty((B, 500), dtype=torch.int32, device=DEV); cnt = torch.empty((B,), dtype=torch.int32, device=DEV)
    rois = torch.empty((B, 500, 4), dtype=torch.float32, device=DEV)
    for unit in (0, 1):
        _lib.check(lib.frr_nms_sorted_indirect(d_src.data_ptr(), N, d_ord.data_ptr(), d_cnt.data_ptr(), B, k, 0.7, 500,
                                               keep.data_ptr(), cnt.data_ptr(), rois.data_ptr(), 0, unit,
                                               torch.cuda.current_stream().cuda_stream), "frr_nms_sorted_indirect")
        assert torch.equal(keep, want_keep) and torch.equal(cnt, want_cnt) and torch.equal(rois, want_rois)


def test_rpn_head_views_zero_copy_in_channels_last(oracle):
    """models/model.py:79-83 hand-off: with channels_last conv outputs the [B,N,2] / [B,N,4] views alias the conv
    outputs (no permute copy) and feed the proposal layer with the same result as the reference's copy path."""
    from faster_rcnn_pytorch_b200 import region
    torch.manual_seed(0)
    B, A, hw = 2, 9, (160, 256)
    H, W = hw[0] // 16, hw[1] // 16
    x = torch.randn(B, 64, H, W, device=DEV)
    cls_conv = torch.nn.Conv2d(64, 2 * A, 1).to(DEV)
    reg_conv = torch.nn.Conv2d(64, 4 * A, 1).to(DEV)
    with torch.no_grad():
        ref_cls = cls_conv(x).permute(0, 2, 3, 1).contiguous().view(B, -1, 2)        # the reference's path
        ref_reg = reg_conv(x).permute(0, 2, 3, 1).contiguous().view(B, -1, 4)
        xcl = x.contiguous(memory_format=torch.channels_last)
        cm = cls_conv.to(memory_format=torch.channels_last)(xcl)
        rm = reg_conv.to(memory_format=torch.channels_last)(xcl)
    assert cm.is_contiguous(memory_format=torch.channels_last)
    cls, reg = region.rpn_head_views(cm, rm)
    assert cls.data_ptr() == cm.data_ptr() and reg.data_ptr() == rm.data_ptr()        # zero copy
    assert cls.shape == (B, H * W * A, 2) and reg.shape == (B, H * W * A, 4)
    torch.testing.assert_close(cls, ref_cls, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(reg, ref_reg, rtol=1e-4, atol=1e-5)
    c2, r2 = region.rpn_head_views(cls_conv(x).contiguous(), reg_conv(x).contiguous())     # NCHW: copy fallback
    torch.testing.assert_close(c2, ref_cls, rtol=1e-4, atol=1e-5)
    rois, cnt = region.rpn_proposals(cls, reg * 0.1, image_hw=hw, mode="test")
    rois2, cnt2 = region.rpn_proposals(cls.clone(), (reg * 0.1).clone(), image_hw=hw, mode="test")
    assert torch.equal(rois, rois2) and torch.equal(cnt, cnt2)


# ------------------------------------------------------------------------------------ FPN-variant proposal layer
@pytest.mark.parametrize("name,mode", [("train", "train"), ("test", "test")])
def test_fpn_variant_proposals_reference_goldens(oracle, name, mode):
    """models/new_model.py:46-83 (torchvision 5-level anchors, min_size 10/1000, 4000|2000 -> 1000): the reference's own
    fp32 boxes / scores -> GPU top-k -> GPU NMS == the reference's keep list; decode within 1e-5."""
    from faster_rcnn_pytorch_b200 import modules
    g = golden("proposal_fpn")
    pre_k, post_k = (4000, 1000) if mode == "train" else (2000, 1000)
    min_size = float(np.float32(10 / 1000))
    boxes, scores, valid = ops.rpn_decode(dev(g[f"{name}_reg"][None]), dev(g[f"{name}_score"][None]),
                                          anchors=dev(g[f"{name}_anchor"]), min_size=min_size)
    np.testing.assert_allclose(boxes[0].cpu().numpy(), g[f"{name}_boxes"], rtol=RTOL, atol=1e-6)
    assert np.array_equal(valid[0].cpu().numpy().astype(bool), oracle.min_size_mask(boxes[0].cpu().numpy(), 10.0))
    r = ops.topk_desc(dev(g[f"{name}_score"][None]), pre_k, valid=dev(g[f"{name}_valid"][None].astype(np.uint8)),
                      boxes=dev(g[f"{name}_boxes"][None]), want_cidx=True)
    n = int(r["count"][0])
    assert np.array_equal(r["cidx"][0, :n].cpu().numpy(), g[f"{name}_topk_idx"])
    keep, cnt, rois = ops.nms_sorted(r["boxes"], 0.7, max_keep=post_k, counts=r["count"], unit_boxes=True)
    k = keep[0, :int(cnt[0])].cpu().numpy()
    assert np.array_equal(k, g[f"{name}_keep"])
    assert np.array_equal(rois[0, :len(k)].cpu().numpy(), g[f"{name}_rois"])
    # the drop-in call (logits in, ragged rois out) runs the same kernels end to end
    out = modules.fpn.region_proposal(dev(g[f"{name}_cls"]), dev(g[f"{name}_reg"]), dev(g[f"{name}_anchor"]), mode)
    assert out.shape[1] == 4 and 0 < out.shape[0] <= post_k


@pytest.mark.parametrize("key", ["128x192", "160x160", "800x1344", "800x1333", "600x1000", "97x131"])
def test_fpn_variant_anchors_generated_on_the_device(oracle, key):
    """models/new_model.py:43-44: torchvision's 5-level AnchorGenerator + the division by (w,h,w,h) as one kernel -- bit
    exact vs the reference's own arrays (sha256 goldens; non-divisible sizes give per-axis integer strides)."""
    from faster_rcnn_pytorch_b200 import modules
    g = golden("anchors_fpn")
    h, w = map(int, key.split("x"))
    hws = [(-(-h // s), -(-w // s)) for s in (4, 8, 16, 32, 64)]
    a = ops.anchors_pyramid(hws, (h, w), DEV).cpu().numpy()
    assert a.shape[0] == int(g[f"n_{key}"])
    assert np.array_equal(sha(a), g[f"sha_{key}"])
    assert np.array_equal(a, oracle.tv_anchors_pyramid(hws, (h, w)))
    gen = modules.fpn.AnchorGenerator()
    t1 = gen((h, w), hws, DEV)
    assert t1 is gen((h, w), hws, DEV) and np.array_equal(t1.cpu().numpy(), a)          # cached per shape


def test_fpn_variant_region_proposal_generates_its_anchors(oracle):
    """fpn.region_proposal without an anchor argument == with the reference's anchor tensor."""
    from faster_rcnn_pytorch_b200 import modules
    g = golden("proposal_fpn")
    hw = (128, 192)
    hws = [(-(-hw[0] // s), -(-hw[1] // s)) for s in (4, 8, 16, 32, 64)]
    a = modules.fpn.region_proposal(dev(g["train_cls"]), dev(g["train_reg"]), dev(g["train_anchor"]), "train")
    b = modules.fpn.region_proposal(dev(g["train_cls"]), dev(g["train_reg"]), None, "train", image_hw=hw, feature_hws=hws)
    assert torch.equal(a, b) and a.shape[0] > 0
    with pytest.raises(ValueError):
        modules.fpn.region_proposal(dev(g["train_cls"]), dev(g["train_reg"]), None, "train")


def test_topk_more_than_65536_anchors_takes_the_general_kernel(oracle):
    """A full-size FPN pyramid (800x1333: 267 069 anchors) is beyond the u16-index fast path."""
    rs = np.random.RandomState(12)
    N, k = 267069, 4000
    scores = synth.unique_scores(rs, N)
    valid = (rs.uniform(size=N) > 0.01)
    r = ops.topk_desc(dev(scores[None]), k, valid=dev(valid[None].astype(np.uint8)), want_cidx=True)
    order, idx = _oracle_topk(oracle, scores, valid, k)
    assert int(r["count"][0]) == k
    assert np.array_equal(r["idx"][0].cpu().numpy(), idx)
    assert np.array_equal(r["cidx"][0].cpu().numpy(), order)


def test_topk_bucket_kernel_hands_over_badly_bucketing_inputs(oracle):
    """The bucket top-k (one histogram pass + per-bucket ranking) hands images whose scores do not bucket well to the radix
    path, which CTA 0 of the image runs in the same launch: all scores equal (empty range), one value repeated far beyond
    the bucket capacity, infinities.  Mixed in one batch with a well-behaved image; every row must equal the oracle's
    order (descending, ties lower index first)."""
    rs = np.random.RandomState(77)
    N, k = 9000, 5000
    rows = [synth.unique_scores(rs, N),                                   # well behaved -> bucket path
            np.full((N,), 0.25, np.float32),                              # empty range
            synth.unique_scores(rs, N), synth.unique_scores(rs, N), synth.unique_scores(rs, N)]
    rows[2][rs.permutation(N)[:3000]] = 0.5                               # 3000 copies of one value (> bucket capacity)
    rows[3][[5, 17]] = np.inf                                             # non-finite: no float bucket map
    rows[3][[6]] = -np.inf
    rows[4] = (rows[4] * 1e-3).astype(np.float32)                          # narrow range, still fine
    rows[4][::2] = rows[4][1]                                             # ... but half of it is one value
    scores = np.stack(rows)
    valid = rs.uniform(size=scores.shape) > 0.05
    r = ops.topk_desc(dev(scores), k, valid=dev(valid.astype(np.uint8)), want_cidx=True)
    cnt = r["count"].cpu().numpy()
    for b in range(len(rows)):
        cidx, idx = _oracle_topk(oracle, scores[b], valid[b], k)
        n = len(idx)
        assert cnt[b] == n
        assert np.array_equal(r["idx"][b, :n].cpu().numpy(), idx), b
        assert np.array_equal(r["cidx"][b, :n].cpu().numpy(), cidx), b
        assert np.array_equal(r["scores"][b, :n].cpu().numpy(), scores[b][idx]), b


def test_proposal_plan_is_cuda_graph_capturable(oracle):
    """frr_rpn_proposals never allocates or synchronises: one call captured into a CUDA graph replays on new inputs and
    gives the same rois / counts as the eager call."""
    from faster_rcnn_pytorch_b200 import region
    hw, B = (320, 480), 3
    ins = [synth.rpn_head_outputs(300 + i, hw) for i in range(B + B)]
    n = synth.num_anchors(hw)
    plan = region.ProposalPlan(B, n, DEV, image_hw=hw, mode="train", logits=False)
    sc = dev(np.stack([x[2] for x in ins[:B]]))
    rg = dev(np.stack([x[1] for x in ins[:B]]))
    graph = plan.capture(sc, rg)
    # new inputs in the captured buffers
    sc.copy_(dev(np.stack([x[2] for x in ins[B:]])))
    rg.copy_(dev(np.stack([x[1] for x in ins[B:]])))
    graph.replay()
    torch.cuda.synchronize()
    got_rois, got_cnt = plan.rois.clone(), plan.count.clone()
    want_rois, want_cnt = region.rpn_proposals(sc, rg, image_hw=hw, mode="train")
    assert torch.equal(got_cnt, want_cnt)
    assert torch.equal(got_rois, want_rois)
    assert int(got_cnt.min()) > 0


@pytest.mark.parametrize("B,N,k", [(1, 21546, 12000), (3, 20646, 6000), (2, 37350, 6000), (5, 3000, 4000)])
def test_topk_cluster_kernel_equals_one_cta_kernel(B, N, k):
    """topk_bucket_kernel on a two-CTA cluster per image (histograms merged through distributed shared memory) against
    one CTA per image: every output identical -- random scores with an invalid mask, heavy ties (quantised scores), all
    scores equal (handed to the radix path by CTA 0 alone), and a batch with empty images."""
    rs = np.random.RandomState(77)
    cases = {
        "random": rs.rand(B, N).astype(np.float32),
        "ties": (rs.randint(0, 500, size=(B, N)) / 500.0).astype(np.float32),
        "equal": np.full((B, N), 0.25, np.float32),
    }
    boxes = dev(rs.rand(B, N, 4).astype(np.float32))
    for name, sc in cases.items():
        valid = (rs.rand(B, N) < 0.9)
        if name == "random" and B > 1:
            valid[B - 1] = False                              # an image without a valid score
        v = dev(valid.astype(np.uint8))
        a = ops.topk_desc(dev(sc), k, valid=v, boxes=boxes, want_cidx=True, ctas_per_image=0)
        b = ops.topk_desc(dev(sc), k, valid=v, boxes=boxes, want_cidx=True, ctas_per_image=1)
        for key in ("count", "idx", "cidx", "scores", "boxes"):
            assert torch.equal(a[key], b[key]), (name, key)
        # and against a stable sort on the host (ties: lower index first)
        for i in range(B):
            src = np.nonzero(valid[i])[0]
            order = src[np.argsort(-sc[i][valid[i]], kind="stable")][:k]
            n = int(a["count"][i])
            assert n == len(order) and np.array_equal(a["idx"][i, :n].cpu().numpy(), order), (name, i)
