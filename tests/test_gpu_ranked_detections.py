"""GPU: the score-ranked evaluation hand-off (ops.pack_detections(rank="score"), frr_pack_detections_ranked) against a
numpy oracle, bit for bit: the class-major rows class_nms keeps, minus the rows past ``per_class_max`` inside their
class, stable-sorted by descending score, the first ``max_det`` scaled and packed like the class-major rows.  The
class-major default is checked to give the first ``max_det`` rows exactly as before."""
import numpy as np
import pytest
import torch

from conftest import golden
from faster_rcnn_pytorch_b200 import _lib, ops, region, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _rows(boxes, scores, labels, wh, xywh):
    """Packed rows of the given detections, in the given order (fp32 arithmetic of pack_row)."""
    sc = np.asarray([wh[0], wh[1], wh[0], wh[1]], np.float32)
    b = (boxes.astype(np.float32) * sc).astype(np.float32)
    if xywh:
        b = np.stack([b[:, 0], b[:, 1], b[:, 2] - b[:, 0], b[:, 3] - b[:, 1]], axis=1)
    return np.concatenate([b, scores[:, None].astype(np.float32), labels[:, None].astype(np.float32)], axis=1)


def oracle_pack(boxes, labels, scores, count, max_det, rank="score", per_class_max=0, image_wh=None, xywh=False):
    """numpy reference of both selections over class-major [B,cap] detections."""
    B, cap = labels.shape
    out = np.zeros((B, max_det, 6), np.float32)
    cnt = np.zeros(B, np.int32)
    for b in range(B):
        n = max(0, min(int(count[b]), cap))
        if rank == "class":
            sel = np.arange(min(n, max_det))
        else:
            keep = np.arange(n)
            if per_class_max > 0:
                seen, ok = {}, np.zeros(n, bool)
                for j in range(n):
                    c = int(labels[b, j])
                    ok[j] = seen.get(c, 0) < per_class_max
                    seen[c] = seen.get(c, 0) + 1
                keep = keep[ok]
            sel = keep[np.argsort(-scores[b, keep], kind="stable")][:max_det]
        wh = image_wh[b] if image_wh is not None else np.ones(2, np.float32)
        out[b, :len(sel)] = _rows(boxes[b, sel], scores[b, sel], labels[b, sel], wh, xywh)
        cnt[b] = len(sel)
    return out, cnt


def check(det, max_det, rank="score", per_class_max=0, image_wh=None, xywh=False, workspace=None):
    db, dl, ds, dc = det
    got, gc = ops.pack_detections(db, dl, ds, dc, max_det, image_wh=None if image_wh is None else dev(image_wh),
                                  xywh=xywh, rank=rank, per_class_max=per_class_max, workspace=workspace)
    want, wc = oracle_pack(db.cpu().numpy(), dl.cpu().numpy(), ds.cpu().numpy(), dc.cpu().numpy(), max_det, rank,
                           per_class_max, image_wh, xywh)
    assert np.array_equal(gc.cpu().numpy(), wc)
    assert np.array_equal(got.cpu().numpy(), want)
    return got, gc


def batch_inputs(seed, B=8, R=300, C=81, ties=False):
    rs = np.random.RandomState(seed)
    prob = np.stack([np.exp(rs.standard_normal((R, C)) * 2) for _ in range(B)])
    prob = (prob / prob.sum(-1, keepdims=True)).astype(np.float32)
    if ties:
        prob = (np.round(prob * 64) / 64).astype(np.float32)   # many equal scores across classes
    boxes = np.stack([synth.random_boxes(seed + 1 + i, R * C, cluster=True)[0].reshape(R, C * 4) for i in range(B)])
    return prob, boxes


RAGGED = np.asarray([300, 0, 17, 300, 150, 1, 299, 64], np.int32)
WH = np.asarray([[1333, 800], [640, 480], [500, 375], [1000, 600], [800, 800], [375, 500], [1, 1], [1920, 1080]],
                np.float32)


@pytest.mark.parametrize("C,seed", [(21, 600), (81, 601)])
@pytest.mark.parametrize("thres", [0.05, 0.005])
def test_ranked_predict_goldens(C, seed, thres):
    """The predict.npz shapes through decode_classwise + class_nms, and the reference's own _suppress output."""
    g = golden("predict")
    cls, reg = synth.head_outputs(seed, 300, C)
    rois, _ = synth.random_boxes(seed + 1, 300)
    prob, boxes = ops.decode_classwise(dev(cls), dev(reg), dev(rois), C)
    det = ops.class_nms(prob[None], boxes[None], C, score_thres=thres, iou_thr=0.3)
    assert int(det[3][0]) > 100                      # more detections than the hand-off keeps
    check(det, 100)
    check(det, 16384, per_class_max=100)             # COCOeval's per-category cap over everything
    check(det, 100, rank="class")

    # identical fp32 inputs to the reference's FRCNN._suppress: rank its own detections
    gb = synth.random_boxes(seed + 2, 300 * C, cluster=False)[0].reshape(1, 300, C * 4)
    det = ops.class_nms(dev(g[f"sup{C}_prob"][None]), dev(gb), C, score_thres=thres, iou_thr=0.3)
    gl, gs, gbb = g[f"sup{C}_label_{thres}"], g[f"sup{C}_score_{thres}"], g[f"sup{C}_bbox_{thres}"]
    assert int(det[3][0]) == len(gl)
    got, gc = check(det, 100)
    top = np.argsort(-gs, kind="stable")[:100]
    assert int(gc[0]) == min(100, len(gl))
    assert np.array_equal(got[0, :len(top)].cpu().numpy(), _rows(gbb[top], gs[top], gl[top], (1.0, 1.0), False))


@pytest.mark.parametrize("per_class_max", [0, 1, 100])
@pytest.mark.parametrize("ties", [False, True])
def test_ranked_batch_ragged(per_class_max, ties):
    """B = 8, ragged roi_count (an image with none), scores tied across classes, pixel scaling with and without xywh."""
    prob, boxes = batch_inputs(700 + ties, ties=ties)
    det = ops.class_nms(dev(prob), dev(boxes), 81, score_thres=0.01, iou_thr=0.3, roi_count=dev(RAGGED))
    counts = det[3].cpu().numpy()
    assert counts[1] == 0 and (counts > 100).sum() >= 3 and ((counts > 0) & (counts < 100)).any()
    ws = ops.pack_ranked_workspace(8, det[1].shape[1], 100, DEV)
    for max_det, wh, xywh in [(100, None, False), (100, WH, True), (37, WH, False), (300, None, True)]:
        check(det, max_det, per_class_max=per_class_max, image_wh=wh, xywh=xywh,
              workspace=ws if max_det == 100 else None)


def test_ranked_capacity_and_counts():
    """class_nms capacity below the detection count, max_det above the capacity, det_count of 0 / below max_det /
    above the capacity."""
    prob, boxes = batch_inputs(800, B=3, C=21, ties=True)
    for cap in (37, 250):
        det = ops.class_nms(dev(prob), dev(boxes), 21, score_thres=0.01, iou_thr=0.3, cap=cap)
        assert (det[3].cpu().numpy() == cap).all()
        for max_det, pcm in [(100, 0), (100, 5), (20, 0), (cap, 3)]:
            check(det, max_det, per_class_max=pcm, image_wh=WH[:3], xywh=True)

    rs = np.random.RandomState(801)
    B, cap = 4, 60
    labels = np.sort(rs.randint(0, 6, (B, cap)), axis=1).astype(np.int32)   # class-major
    scores = (rs.randint(1, 9, (B, cap)) / 8).astype(np.float32)           # ties within and across classes
    bx = rs.uniform(0, 1, (B, cap, 4)).astype(np.float32)
    count = np.asarray([0, 12, cap, cap + 25], np.int32)
    det = (dev(bx), dev(labels), dev(scores), dev(count))
    for max_det, pcm in [(8, 0), (100, 0), (100, 4), (cap, 1)]:
        check(det, max_det, per_class_max=pcm, image_wh=WH[:B])


def test_class_major_default_unchanged():
    """Without the new arguments pack_detections keeps the first max_det class-major rows, as it always did."""
    prob, boxes = batch_inputs(900)
    det = ops.class_nms(dev(prob), dev(boxes), 81, score_thres=0.01, iou_thr=0.3, roi_count=dev(RAGGED))
    db, dl, ds, dc = det
    for max_det, wh, xywh in [(100, WH, True), (100, None, False), (5000, None, False)]:
        a, ac = ops.pack_detections(db, dl, ds, dc, max_det, image_wh=None if wh is None else dev(wh), xywh=xywh)
        want, wc = oracle_pack(db.cpu().numpy(), dl.cpu().numpy(), ds.cpu().numpy(), dc.cpu().numpy(), max_det, "class",
                               0, wh, xywh)
        assert np.array_equal(a.cpu().numpy(), want) and np.array_equal(ac.cpu().numpy(), wc)


def test_ranked_argument_errors():
    prob, boxes = batch_inputs(901, B=1, C=81)
    db, dl, ds, dc = ops.class_nms(dev(prob), dev(boxes), 81, score_thres=0.01)      # cap 300 * 80 > 16384
    with pytest.raises(_lib.FrrError, match="workspace too small"):
        ops.pack_detections(db, dl, ds, dc, 100, rank="score",
                            workspace=torch.empty(16, dtype=torch.uint8, device=DEV))
    with pytest.raises(ValueError, match="16384"):
        ops.pack_detections(db, dl, ds, dc, 16385, rank="score")
    with pytest.raises(ValueError, match="rank"):
        ops.pack_detections(db, dl, ds, dc, 100, rank="area")


def test_infer_plan_ranked_graph_equals_eager():
    """InferPlan(rank="score"): a captured detect graph replayed on new head outputs gives the eager result, and both are
    the ranking of the plan's own class_nms detections."""
    hw, B, NC = (320, 480), 2, 81
    plan = region.InferPlan(B, hw, NC, DEV, score_thres=0.005, rank="score", per_class_max=100)
    fh, fw = plan.fhw
    ins = [synth.rpn_head_outputs(1200 + i, hw) for i in range(B)]
    lg = np.stack([x[0] for x in ins]); rg = np.stack([x[1] for x in ins])
    plan.pool(dev(synth.features(1207, B, 8, fh, fw)), dev(lg), dev(rg))
    heads = [synth.head_outputs(1220 + i, plan.R, NC) for i in range(B)]
    d_hc = dev(np.concatenate([h[0] for h in heads])); d_hr = dev(np.concatenate([h[1] for h in heads]))
    graph, (g_packed, g_count) = region._capture(lambda: plan.detect(d_hc, d_hr), plan.device)

    heads2 = [synth.head_outputs(1240 + i, plan.R, NC) for i in range(B)]
    d_hc.copy_(dev(np.concatenate([h[0] for h in heads2]))); d_hr.copy_(dev(np.concatenate([h[1] for h in heads2])))
    graph.replay()
    eager = plan.detect(d_hc, d_hr, return_all=True)
    torch.cuda.synchronize()
    assert (eager["det"][3].cpu().numpy() > plan.max_det).all()
    assert torch.equal(g_packed, eager["packed"]) and torch.equal(g_count, eager["count"])
    db, dl, ds, dc = (t.cpu().numpy() for t in eager["det"])
    want, wc = oracle_pack(db, dl, ds, dc, plan.max_det, "score", 100)
    assert np.array_equal(g_packed.cpu().numpy(), want) and np.array_equal(g_count.cpu().numpy(), wc)
