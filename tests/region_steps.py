"""A predict step and a training step of the batched region stage written with ``torch.ops.frr.*`` and aten only, so that
``make_fx`` / ``torch.compile(fullgraph=True)`` can trace them whole.  The Fast R-CNN head is one fixed linear layer on
the pooled features.

predict: proposals -> rois5 -> RoIPool -> head -> decode_classwise -> class_nms -> pack_detections(rank="score")
train:   make_targets -> rois5 -> RoIPool -> head -> region_loss (its backward reaches the features through RoIPool)
"""
import torch

from faster_rcnn_pytorch_b200 import ops, region, torch_ops  # noqa: F401  (torch_ops registers torch.ops.frr.*)

frr = torch.ops.frr
STRIDE = 16
NMS_THRESH, MIN_SIZE = region.RPN_NMS_THRESH, ops._MIN_SIZE


def head(pooled, w_cls, w_reg, B, R, NC):
    x = pooled.flatten(1)
    return (x @ w_cls).view(B * R, NC), (x @ w_reg).view(B * R, 4 * NC)


def pool(feat, rois5, image_hw):
    if image_hw is None:
        return frr.roi_pool(feat, rois5, 1.0, 7, 7)[0]
    return frr.roi_pool_sized(feat, rois5, image_hw, 1.0, 7, 7, STRIDE)[0]


def predict(feat, rpn_cls, rpn_reg, image_hw, w_cls, w_reg, *, grid, NC, pre=6000, post=300, max_det=100):
    """``image_hw`` int32 [B,2] device sizes of a batch padded to ``grid`` cells.  Returns (packed [B,max_det,6],
    counts [B], rois [B,post,4], roi counts [B])."""
    B = feat.shape[0]
    rois, cnt = frr.rpn_proposals_sized(rpn_cls, rpn_reg, image_hw, grid[0], grid[1], pre, post, NMS_THRESH, MIN_SIZE)
    r5 = frr.rois5(rois, cnt, grid[0], grid[1], image_hw, STRIDE)
    hc, hr = head(pool(feat, r5, image_hw), w_cls, w_reg, B, post, NC)
    prob, boxes = frr.decode_classwise(hc, hr, rois.reshape(-1, 4), NC)
    db, dl, ds, dc = frr.class_nms(prob.view(B, post, NC), boxes.view(B, post, 4 * NC), NC, 0.05, 0.3, cnt, None)
    packed, pc = frr.pack_detections(db, dl, ds, dc, max_det, None, False, "score", 0)
    return packed, pc, rois, cnt


def train(feat, rpn_cls, rpn_reg, gt, gt_count, gt_label, props, prop_count, mt_state, image_hw, w_cls, w_reg, *, padded_hw,
          NC):
    """Both target makers (device sampling from ``mt_state``, advanced in place), RoIPool of the sampled rois, the head
    and the fused loss.  Returns (loss [B,5], targets, rois5)."""
    B = feat.shape[0]
    fh, fw = padded_hw[0] // STRIDE, padded_hw[1] // STRIDE
    t = frr.make_targets(gt, gt_count, gt_label, props, prop_count, mt_state, padded_hw[0], padded_hw[1], image_hw)
    S = t[4].shape[1]
    r5 = frr.rois5(t[4], t[6], fh, fw, image_hw, STRIDE)
    hc, hr = head(pool(feat, r5, image_hw), w_cls, w_reg, B, S, NC)
    loss = frr.region_loss(rpn_cls, rpn_reg, t[0], t[1], hc.view(B, S, NC), hr.view(B, S, 4 * NC), t[2], t[3])[0]
    return loss, t, r5


def train_grads(feat, rpn_cls, rpn_reg, *args, **kw):
    """``train`` and the gradients of the summed totals w.r.t. the features and the RPN head outputs."""
    loss, t, r5 = train(feat, rpn_cls, rpn_reg, *args, **kw)
    return (loss,) + torch.autograd.grad(loss[:, 0].sum(), (feat, rpn_cls, rpn_reg))
