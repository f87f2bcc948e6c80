"""The target makers (csrc/targets.cu) at every launch geometry they select: the RPN assign kernel's cluster of
S = 8 / 4 / 2 / 1 CTAs per image and the finalize kernel's slab count, computed here from the rule in targets.cu and
observed in the profiler trace.  IoU row max, argmax, pre-sampling labels, counts and the order of the positive and
negative lists are compared bit for bit with the oracle; encode() with float64 under a per-component bound.  Also:
per-GT ties that straddle two CTAs' slabs, IoUs exactly on the 0.7f / 0.3f / 0.5f thresholds and one ulp off them,
the largest Gmax the shared-memory check accepts (and Gmax + 1 refused before any launch), the Fast R-CNN maker at
R = 0 / 12 000, ragged counts, short samples and label offsets 0 / 1, and degenerate GT boxes."""
import json

import numpy as np
import pytest
import torch

import training_refs as tr
from faster_rcnn_pytorch_b200 import _lib, ops, synth, targets

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
f32 = np.float32
STD = np.asarray([0.1, 0.1, 0.2, 0.2], f32)       # models/model.py:174-177
SMEM_LIMIT = 227 * 1024


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def cluster_size(B, N):
    """launch_rpn_assign: one CTA per ~2048 anchors, at most 8, no more than ~2 CTAs per SM for the batch."""
    S = 1
    while S < 8 and N >= 2048 * (S * 2) and B * (S * 2) <= 2 * sms():
        S *= 2
    return S


def finalize_slabs(B, N):
    s = 1
    while s < 16 and N >= 2048 * (s * 2) and B * (s * 2) <= 2 * sms():
        s *= 2
    return s


def rpn_smem(G, N, S):
    cpc = ((N + 31) // 32 + S - 1) // S
    return 256 + G * 16 + ((G + 1) & ~1) * 4 + 10 * G * 8 + 2 * cpc * 4 + 16


def frcnn_smem(G, M):
    return 256 + G * 16 + ((G + 3) & ~3) * 4 + 2 * ((M + 31) // 32) * 4 + 16


def presample(oracle, gt, anchors, variant="vgg"):
    """The assign kernel's outputs for one image from the oracle's fp32 IoU (models/model.py:196-216 and
    new_model.py:309-318): iou_max, argmax, label8 (-2 outside the image, else -1 / 0 / 1 before sampling)."""
    fpn = variant == "fpn"
    inside = np.ones(len(anchors), bool) if fpn else (
        (anchors[:, 0] >= 0) & (anchors[:, 1] >= 0) & (anchors[:, 2] <= 1) & (anchors[:, 3] <= 1))
    iou = oracle.pairwise_iou_eps(anchors[inside], gt, 0.0 if fpn else 1e-5)
    mx, am = iou.max(1), iou.argmax(1)
    lab = np.full(len(mx), -1, np.int8)
    lab[mx < f32(0.3)] = 0
    if fpn:
        lab[(iou == iou.max(0)[None, :]).any(1)] = 1
    else:
        lab[iou.argmax(0)] = 1
    lab[mx >= f32(0.7)] = 1
    im, amf, l8 = np.zeros(len(anchors), f32), np.zeros(len(anchors), np.int32), np.full(len(anchors), -2, np.int8)
    im[inside], amf[inside], l8[inside] = mx, am, lab
    return im, amf, l8


def check_assign(ws, b, want, what):
    im, am, l8 = want
    # bit for bit up to the sign of a zero: the row max of -0.0 (0 over the negative union of a GT inverted in one axis)
    # and +0.0 may be either zero in the reference's max and in the kernel, and no label depends on it
    got = ws["iou_max"][b].cpu().numpy() + f32(0)
    assert np.array_equal(got.view(np.uint32), (im + f32(0)).view(np.uint32)), f"{what}: iou_max"
    assert np.array_equal(ws["argmax"][b].cpu().numpy(), am), f"{what}: argmax"
    assert np.array_equal(ws["label8"][b].cpu().numpy(), l8), f"{what}: label8"
    pos, neg = np.nonzero(l8 == 1)[0], np.nonzero(l8 == 0)[0]
    assert tuple(ws["counts"][b].cpu().numpy()) == (len(pos), len(neg)), f"{what}: counts"
    assert np.array_equal(ws["pos_list"][b, :len(pos)].cpu().numpy(), pos), f"{what}: positive list order"
    assert np.array_equal(ws["neg_list"][b, :len(neg)].cpu().numpy(), neg), f"{what}: negative list order"


def kernel_grids(fn, tmp_path):
    """Run ``fn`` under torch.profiler and return {kernel name: [grid of each launch]} from the exported trace."""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    grids = {}
    for e in json.loads(path.read_text())["traceEvents"]:
        if e.get("cat") == "kernel":
            grids.setdefault(e["name"], []).append(e.get("args", {}).get("grid"))
    return out, grids


def grid_of(grids, name):
    hits = [g for k, v in grids.items() if name in k and "sized" not in k for g in v]
    assert len(hits) == 1, (name, list(grids))
    return hits[0]


GEOMETRY = [((600, 1000), 1), ((600, 1000), 37), ((600, 1000), 38), ((600, 1000), 64), ((600, 1000), 75),
            ((600, 1000), 148), ((600, 1000), 149), ((800, 1333), 9)]


@pytest.mark.parametrize("hw,B", GEOMETRY, ids=[f"{h}x{w}-B{b}" for (h, w), b in GEOMETRY])
def test_rpn_targets_every_cluster_size_vs_oracle(oracle, tmp_path, hw, B):
    anchors = oracle.enumerate_anchors(hw)
    N = len(anchors)
    S, slabs = cluster_size(B, N), finalize_slabs(B, N)
    if sms() == 148:                                   # the geometry the batch sizes were chosen for (B200)
        want_s = {1: 8, 37: 8, 38: 4, 64: 4, 75: 2, 148: 2, 149: 1, 9: 8}[B]
        assert S == want_s and (N != 37350 or slabs == 16)
    G = 12
    cnt = np.asarray([1 + (7 * i) % G for i in range(B)], np.int32)          # ragged GT counts
    gts = np.zeros((B, G, 4), f32)
    for i in range(B):
        gts[i, :cnt[i]] = synth.gt_boxes(7000 + i, int(cnt[i]))[0]

    def go():
        ws = ops.rpn_targets_assign(dev(gts), dev(cnt), N, image_hw=hw)
        return ws, ops.rpn_targets_finalize(ws)
    (ws, (labels, reg)), grids = kernel_grids(go, tmp_path)
    # the launch geometry, observed
    assert grid_of(grids, "rpn_assign_kernel") == [B * S, 1, 1]
    assert grid_of(grids, "rpn_finalize_kernel") == [slabs, B, 1]
    labels, reg = labels.cpu().numpy(), reg.cpu().numpy()
    for i in range(B):
        g = gts[i, :cnt[i]]
        want = presample(oracle, g, anchors)
        check_assign(ws, i, want, f"image {i}")
        l8 = want[2]
        assert np.array_equal(labels[i], np.where(l8 == -2, -1, l8).astype(np.int64))
        ins = l8 != -2
        assert not reg[i][~ins].any()
        tr.check_encode(reg[i][ins], g[want[1][ins]], anchors[ins], what="rpn encode")


@pytest.mark.parametrize("variant", ["vgg", "fpn"])
@pytest.mark.parametrize("B", [1, 38, 75, 149])
def test_rpn_per_gt_ties_across_slabs(oracle, variant, B):
    """Each GT's best IoU is reached, bit for bit, by the last anchor of slab r - 1 and the first of slab r: the VGG
    maker labels the lower index only (first argmax, through the cluster's distributed-shared-memory exchange), the
    FPN maker both (torch.where(iou == max))."""
    N = 20646
    S = cluster_size(B, N)
    anchors, gt, ties = tr.slab_tie_case(N, max(S, 2), variant)
    gts = np.repeat(gt[None], B, 0)
    ws = ops.rpn_targets_assign(dev(gts), None, N, anchors=dev(anchors), variant=variant)
    want = presample(oracle, gt, anchors, variant)
    for i in sorted({0, B // 2, B - 1}):
        check_assign(ws, i, want, f"image {i}")
    l8 = ws["label8"][B - 1].cpu().numpy()
    for lo, hi in ties:
        assert l8[lo] == 1 and l8[hi] == (1 if variant == "fpn" else -1), (lo, hi, l8[lo], l8[hi])


CASES_THR = [(0.7, -1, -1), (0.7, 0, 1), (0.7, 1, 1), (0.3, -1, 0), (0.3, 0, -1), (0.3, 1, -1)]


def test_rpn_labels_on_the_iou_thresholds(oracle):
    """IoU exactly 0.7f / 0.3f and one ulp either side: >= 0.7 positive, < 0.3 negative, in between ignored.  A copy of
    the GT is the GT's best anchor, so the pair's label comes from the thresholds alone."""
    B = len(CASES_THR)
    rs = np.random.RandomState(3)
    fill = rs.uniform(0.9, 0.98, (62, 2)).astype(f32)
    fill = np.concatenate([fill, fill + f32(0.01)], 1)
    for b, (t, side, lab) in enumerate(CASES_THR):
        box, gt = tr.threshold_pair(t, side)
        anchors = np.concatenate([box[None], gt[None], fill]).astype(f32)
        ws = ops.rpn_targets_assign(dev(gt[None, None]), None, len(anchors), anchors=dev(anchors))
        want = presample(oracle, gt[None], anchors)
        check_assign(ws, 0, want, f"threshold {t} side {side}")
        assert int(ws["label8"][0, 0]) == lab, (t, side)
        assert (ws["iou_max"][0, 0].item() >= f32(t)) == (side >= 0)


def test_frcnn_labels_on_the_fg_threshold(oracle):
    """Fast R-CNN: IoU >= 0.5f foreground, below it background, at 0.5f exactly and one ulp either side."""
    for side, lab in ((-1, 0), (0, 1), (1, 1)):
        box, gt = tr.threshold_pair(0.5, side)
        ws = ops.frcnn_targets_assign(dev(box[None, None]), None, dev(gt[None, None]), None)
        w = oracle.pairwise_iou_eps(np.concatenate([box[None], gt[None]]), gt[None])[:, 0]
        assert np.array_equal(ws["iou_max"][0].cpu().numpy().view(np.uint32), w.view(np.uint32))
        assert ws["label8"][0].cpu().numpy().tolist() == [lab, 1]


def _max_gmax(smem):
    g = 1
    while smem(g + 1) <= SMEM_LIMIT:
        g += 1
    return g


@pytest.mark.parametrize("G", [1, 160, 1000, "max"])
def test_rpn_assign_gmax_up_to_the_shared_memory_limit(oracle, G):
    hw = (160, 256)
    anchors = oracle.enumerate_anchors(hw)
    N = len(anchors)
    S = cluster_size(1, N)
    gmax = _max_gmax(lambda g: rpn_smem(g, N, S))
    assert 2000 < gmax < 2500
    G = gmax if G == "max" else G
    gt = synth.gt_boxes(G, G)[0]
    ws = ops.rpn_targets_assign(dev(gt[None]), None, N, image_hw=hw)
    check_assign(ws, 0, presample(oracle, gt, anchors), f"G={G}")
    if G == gmax:
        big = synth.gt_boxes(1, G + 1)[0]
        before = _lib.launch_count()
        with pytest.raises(ValueError, match="shared memory"):
            ops.rpn_targets_assign(dev(big[None]), None, N, image_hw=hw)
        assert _lib.launch_count() == before


@pytest.mark.parametrize("G", [1, 160, 1000, "max"])
def test_frcnn_assign_gmax_up_to_the_shared_memory_limit(oracle, G):
    R = 2000
    gmax = _max_gmax(lambda g: frcnn_smem(g, R + g))
    G = gmax if G == "max" else G
    gt = synth.gt_boxes(G + 1, G)[0]
    rois = synth.random_boxes(5, R)[0]
    ws = ops.frcnn_targets_assign(dev(rois[None]), None, dev(gt[None]), None)
    rows = np.concatenate([rois, gt])
    pick = np.unique(np.concatenate([np.arange(0, R + G, max(1, (R + G) // 700)), [R + G - 1]]))
    iou = oracle.pairwise_iou_eps(rows[pick], gt)
    assert np.array_equal(ws["iou_max"][0].cpu().numpy()[pick].view(np.uint32), iou.max(1).view(np.uint32))
    assert np.array_equal(ws["argmax"][0].cpu().numpy()[pick], iou.argmax(1))
    if G == gmax:
        before = _lib.launch_count()
        with pytest.raises(ValueError, match="shared memory"):
            ops.frcnn_targets_assign(dev(rois[None]), None, dev(synth.gt_boxes(2, G + 1)[0][None]), None)
        assert _lib.launch_count() == before


FRCNN_CASES = [("r0", [0, 0], [3, 1], "vgg"), ("r12000", [12000, 11000], [8, 40], "vgg"),
               ("ragged_short", [2000, 30, 3, 500], [8, 1, 2, 5], "vgg"), ("fpn_offset0", [12000, 7, 0], [5, 2, 9], "fpn")]


@pytest.mark.parametrize("name,rc,gc,variant", FRCNN_CASES, ids=[c[0] for c in FRCNN_CASES])
def test_frcnn_targets_counts_and_offsets_vs_oracle(oracle, name, rc, gc, variant):
    """Labels + label_offset (1 for the VGG maker, 0 for the FPN one), sampled rows and keep indices bit-exact; encode
    divided by std within the float64 bound; rows past a short sample padded."""
    B, R, G = len(rc), max(rc), max(gc)
    rois = np.zeros((B, R, 4), f32)
    gts = np.zeros((B, G, 4), f32)
    labs = np.zeros((B, G), np.int64)
    for i in range(B):
        rois[i, :rc[i]] = synth.random_boxes(300 + i, rc[i])[0] if rc[i] else np.zeros((0, 4), f32)
        b, l = synth.gt_boxes(400 + i, gc[i])
        gts[i, :gc[i]], labs[i, :gc[i]] = b, l
    cls, reg, srois, kidx, n = targets.frcnn_targets(dev(rois), dev(np.asarray(rc, np.int32)), dev(gts),
                                                     dev(np.asarray(gc, np.int32)), dev(labs),
                                                     randperm=oracle.HostRandperm(55), variant=variant)
    rp = oracle.HostRandperm(55)
    cls, reg, srois = cls.cpu().numpy(), reg.cpu().numpy(), srois.cpu().numpy()
    for i in range(B):
        w = oracle.frcnn_targets(gts[i, :gc[i]], labs[i, :gc[i]], rois[i, :rc[i]], rp, variant=variant)
        k = len(w["keep"])
        assert int(n[i]) == k
        assert np.array_equal(cls[i, :k], w["cls"]) and (cls[i, k:] == -1).all()
        assert np.array_equal(kidx[i, :k].cpu().numpy().astype(np.int64), w["keep"])
        assert np.array_equal(srois[i, :k], w["sample_rois"])
        g = gts[i, :gc[i]][w["argmax"][w["keep"]]]
        tr.check_encode(reg[i, :k], g, w["sample_rois"], STD, what="frcnn encode")
        assert not reg[i, k:].any()


def test_frcnn_finalize_divides_each_component_by_its_std():
    """The maker's std has equal z and w components; with four different ones each encoded component must be divided by
    its own.  Positions are selected in list order (no draw), so the expected rows follow from the assign lists."""
    rois = synth.random_boxes(31, 500)[0]
    gt, lab = synth.gt_boxes(32, 6)
    ws = ops.frcnn_targets_assign(dev(rois[None]), None, dev(gt[None]), None)
    n_pos, n_neg = (int(v) for v in ws["counts"][0].cpu())
    kp = min(n_pos, 32)
    kn = min(n_neg, 128 - kp)
    sel = np.zeros((1, 128), np.int32)
    sel[0, :kp], sel[0, kp:kp + kn] = np.arange(kp), np.arange(kn)
    std = np.asarray([0.1, 0.2, 0.3, 0.4], f32)
    cls, reg, srois, kidx = ops.frcnn_targets_finalize(ws, dev(lab[None]), dev(sel), dev(np.asarray([[kp, kp + kn]], np.int32)),
                                                       std=std)
    k = kp + kn
    idx = kidx[0, :k].cpu().numpy()
    assert np.array_equal(idx, np.concatenate([ws["pos_list"][0, :kp].cpu().numpy(), ws["neg_list"][0, :kn].cpu().numpy()]))
    rows = np.concatenate([rois, gt])
    am = ws["argmax"][0].cpu().numpy()
    assert np.array_equal(cls[0, :kp].cpu().numpy(), lab[am[idx[:kp]]] + 1) and not cls[0, kp:k].cpu().any()
    tr.check_encode(reg[0, :k].cpu().numpy(), gt[am[idx]], rows[idx], std, what="frcnn encode")


DEGENERATE = {"zero_width": [0.3, 0.3, 0.3, 0.6], "zero_height": [0.3, 0.3, 0.6, 0.3],
              "inverted_x": [0.7, 0.1, 0.1, 0.9], "inverted_y": [0.1, 0.7, 0.9, 0.1], "inverted_both": [0.8, 0.8, 0.2, 0.2]}


@pytest.mark.parametrize("kind", list(DEGENERATE))
def test_rpn_targets_degenerate_gt_boxes(oracle, kind):
    """A GT box of zero width / height, or inverted in one or both axes, next to a normal one.  Anchor 0 is larger than
    the inverted boxes' |area| and anchor 1 smaller, so an inverted-in-one-axis GT has IoU +0.0 with anchor 0 and -0.0
    (0 over a negative union) with anchor 1: the reference's argmax treats the two zeros as equal and takes anchor 0."""
    bad = np.asarray(DEGENERATE[kind], f32)
    gt = np.stack([bad, np.asarray([0.05, 0.05, 0.35, 0.4], f32)])
    rs = np.random.RandomState(9)
    fill = rs.uniform(0.9, 0.98, (200, 2)).astype(f32)
    anchors = np.concatenate([[[0.0, 0.0, 1.0, 1.0], [0.9, 0.9, 0.95, 0.95]], np.concatenate([fill, fill + f32(0.01)], 1)])
    anchors = anchors.astype(f32)
    ws = ops.rpn_targets_assign(dev(gt[None]), None, len(anchors), anchors=dev(anchors))
    want = presample(oracle, gt, anchors)
    check_assign(ws, 0, want, kind)
    labels, reg = targets.rpn_targets(dev(gt[None]), None, anchors=dev(anchors), randperm=oracle.HostRandperm(4))
    w = oracle.rpn_targets(gt, anchors, oracle.HostRandperm(4))
    assert np.array_equal(labels[0].cpu().numpy(), w["labels"])
    reg = reg[0].cpu().numpy()
    tr.check_encode(reg, gt[w["argmax"]], anchors, what=f"{kind} encode")
    if kind in ("zero_width", "zero_height"):
        col = 2 if kind == "zero_width" else 3
        hit = w["argmax"] == 0
        assert hit.any() and (reg[hit, col] == -np.inf).all()


def test_rpn_targets_inverted_gt_in_a_batch_at_full_size(oracle):
    """The inverted-GT case through generated anchors at 600 x 1000, in a batch that runs 8-CTA clusters."""
    hw = (600, 1000)
    anchors = oracle.enumerate_anchors(hw)
    small = float((anchors[:, 2] - anchors[:, 0]).min() * (anchors[:, 3] - anchors[:, 1]).min())
    gts = np.stack([np.stack([synth.gt_boxes(20 + i, 3)[0][0], np.asarray([0.6, 0.2, 0.2, 0.2 + 4 * small / 0.4], f32),
                              synth.gt_boxes(20 + i, 3)[0][2]]) for i in range(4)]).astype(f32)
    ws = ops.rpn_targets_assign(dev(gts), None, len(anchors), image_hw=hw)
    for i in range(4):
        check_assign(ws, i, presample(oracle, gts[i], anchors), f"image {i}")


@pytest.fixture(scope="module", autouse=True)
def _report_worst_ratios():
    yield
    print("\nworst error/bound ratios (targets):", {k: round(v, 4) for k, v in sorted(tr.WORST.items())})
