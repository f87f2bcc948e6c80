"""Drop-in replacements for the reference's region-stage call sites (models/model.py:6-9,288-298).

Same class names, constructor arguments, forward signatures, return types and error behaviour as the
reference modules, single image per call like the reference; every computation is a libfrr kernel.  The
batched, sync-free entry points are in ``region.py`` / ``targets.py``.

    from faster_rcnn_pytorch_b200.modules import nms, RoIPool, RegionProposal, RPNTargetMaker, FastRcnnTargetMaker
    from faster_rcnn_pytorch_b200.anchor import FRCNNAnchorMaker
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn

from . import ops, region, targets

__all__ = ["nms", "roi_pool", "roi_align", "RoIPool", "RoIAlign", "MultiScaleRoIAlign", "RegionProposal", "RPNTargetMaker",
           "FastRcnnTargetMaker", "predict_tail", "suppress", "fpn", "RPNLoss", "FastRCNNLoss", "FRCNNLoss"]

roi_pool = ops.roi_pool
roi_align = ops.roi_align


def _as_anchor_tensor(anchor, device):
    if isinstance(anchor, np.ndarray):
        anchor = torch.from_numpy(anchor)
    return anchor.to(device=device, dtype=torch.float32).contiguous()


def nms(boxes: torch.Tensor, scores: torch.Tensor, iou_threshold: float) -> torch.Tensor:
    """Drop-in for ``torchvision.ops.nms`` (models/model.py:53,394): int64 indices of the kept boxes, sorted by
    decreasing score; ties keep the lower index first (stable), IoU compared in double like the CPU kernel."""
    if boxes.dim() != 2 or boxes.shape[1] != 4 or scores.dim() != 1 or scores.shape[0] != boxes.shape[0]:
        raise RuntimeError("nms: boxes must be [n,4] and scores [n]")
    n = boxes.shape[0]
    if n == 0:
        return torch.empty((0,), dtype=torch.int64, device=boxes.device)
    b = boxes.detach().to(torch.float32).contiguous()
    if n > 16384:
        # beyond the in-shared-memory sort of frr_topk_desc_opt (the reference never passes more than 12000 boxes,
        # models/model.py:24-28): the ordering falls to torch's stable device sort, the NMS itself stays frr_nms_sorted
        order = torch.argsort(scores.detach().to(torch.float32), descending=True, stable=True)
        keep, cnt, _ = ops.nms_sorted(b.index_select(0, order).reshape(1, n, 4), float(iou_threshold), gather=False)
        return order.index_select(0, keep[0, :int(cnt[0])].to(torch.int64))
    top = ops.topk_desc(scores.detach().to(torch.float32).reshape(1, n), n, boxes=b.reshape(1, n, 4))
    keep, cnt, _ = ops.nms_sorted(top["boxes"], float(iou_threshold), gather=False)
    k = int(cnt[0])
    return top["idx"][0].index_select(0, keep[0, :k].to(torch.int64)).to(torch.int64)


class RoIPool(nn.Module):
    """Drop-in for ``torchvision.ops.RoIPool`` (models/model.py:97)."""

    def __init__(self, output_size, spatial_scale: float):
        super().__init__()
        self.output_size = output_size
        self.spatial_scale = spatial_scale

    def forward(self, input, rois):
        return ops.roi_pool(input, rois, self.output_size, self.spatial_scale)


class RoIAlign(nn.Module):
    """Drop-in for ``torchvision.ops.RoIAlign`` (the 7x7, sampling_ratio=2 pooler of models/new_model.py:127)."""

    def __init__(self, output_size, spatial_scale: float, sampling_ratio: int, aligned: bool = False):
        super().__init__()
        self.output_size, self.spatial_scale = output_size, spatial_scale
        self.sampling_ratio, self.aligned = sampling_ratio, aligned

    def forward(self, input, rois):
        return ops.roi_align(input, rois, self.output_size, self.spatial_scale, self.sampling_ratio, self.aligned)


class MultiScaleRoIAlign(nn.Module):
    """Drop-in for ``torchvision.ops.MultiScaleRoIAlign(featmap_names, output_size, sampling_ratio)`` as constructed at
    models/new_model.py:127 and called at :143 with ``(features: dict, boxes: list[Tensor[L,4]], image_shapes)``."""

    def __init__(self, featmap_names, output_size, sampling_ratio, *, canonical_scale: int = 224, canonical_level: int = 4):
        super().__init__()
        self.featmap_names = list(featmap_names)
        self.output_size = (output_size, output_size) if isinstance(output_size, int) else tuple(output_size)
        self.sampling_ratio = sampling_ratio
        self.canonical_scale, self.canonical_level = canonical_scale, canonical_level

    def forward(self, x, boxes, image_shapes):
        feats = [v for k, v in x.items() if k in self.featmap_names]      # TV ops/poolers.py _filter_input
        return ops.multiscale_roi_align(feats, boxes, image_shapes, self.output_size, self.sampling_ratio,
                                        float(self.canonical_scale), int(self.canonical_level))


class RegionProposal(nn.Module):
    """models/model.py:12-58.  ``forward(cls [N,2], reg [N,4], anchor [N,4], mode)`` -> rois [<=2000|300, 4]."""

    def __init__(self):
        super().__init__()
        self.min_size = 1

    def forward(self, cls, reg, anchor, mode):
        if mode not in region.PROPOSAL_MODES:
            mode = "train"          # the reference only special-cases 'test' (:26)
        anchor = _as_anchor_tensor(anchor, reg.device)
        rois, count = region.rpn_proposals(cls.detach().unsqueeze(0).to(torch.float32), reg.detach().unsqueeze(0).to(torch.float32),
                                           anchors=anchor, mode=mode)
        return rois[0, :int(count[0])]     # ragged like the reference: one host sync


class RPNTargetMaker(nn.Module):
    """models/model.py:182-266.  ``forward(bbox [G,4], anchor [N,4])`` -> (rpn_tg_cls int64 [N], rpn_tg_reg [N,4])."""

    def __init__(self):
        super().__init__()

    def forward(self, bbox, anchor):
        anchor = _as_anchor_tensor(anchor, bbox.device)
        labels, reg = targets.rpn_targets(bbox.detach().to(torch.float32).reshape(1, -1, 4), None, anchors=anchor)
        return labels[0], reg[0]


class FastRcnnTargetMaker(nn.Module):
    """models/model.py:123-179.  ``forward(bbox [list of [G,4]], label [list of [G]], rois [R,4])`` ->
    (fast_rcnn_tg_cls int64 [<=128], fast_rcnn_tg_reg [<=128,4], sample_rois [<=128,4])."""

    def __init__(self):
        super().__init__()

    def forward(self, bbox, label, rois):
        bbox = bbox[0]      # remove the list for batch (:130-131)
        label = label[0]
        cls, reg, srois, _, n = targets.frcnn_targets(rois.detach().to(torch.float32).unsqueeze(0), None,
                                                      bbox.detach().to(torch.float32).unsqueeze(0), None,
                                                      label.detach().to(torch.int64).unsqueeze(0))
        k = int(n[0])
        return cls[0, :k], reg[0, :k], srois[0, :k]


class fpn:
    """Drop-ins for the target makers of the FPN variant, models/new_model.py (what main.py trains today).  Same class
    names and forward signatures as there (tensors, not per-image lists); normalised xyxy boxes like the reference."""

    PROPOSAL_MODES = {"train": (4000, 1000), "test": (2000, 1000)}   # models/new_model.py:52-56
    MIN_SIZE = float(np.float32(10 / 1000))                          # models/new_model.py:21,66 (fp32 compare)

    class AnchorGenerator:
        """Drop-in for the two anchor lines of ``RegionProposalNetwork.forward`` (models/new_model.py:43-44):
        ``torchvision...AnchorGenerator(sizes, aspect_ratios)(ImageList(x, ...), features)[0] / (w, h, w, h)``, generated
        by one kernel on the device and cached per (image size, pyramid shape, device)."""

        def __init__(self, sizes=((32,), (64,), (128,), (256,), (512,)), aspect_ratios=((0.5, 1.0, 2.0),) * 5):
            if any(len(s) != 1 for s in sizes) or any(tuple(a) != tuple(aspect_ratios[0]) for a in aspect_ratios):
                raise ValueError("AnchorGenerator: one size per level and the same aspect ratios on every level "
                                 "(the configuration of models/new_model.py:23-25)")
            self.sizes = tuple(float(s[0]) for s in sizes)
            self.aspect_ratios = tuple(float(a) for a in aspect_ratios[0])
            self._cache = {}

        def __call__(self, image_hw, feature_hws, device):
            key = (tuple(image_hw), tuple(tuple(x) for x in feature_hws), str(device))
            if key not in self._cache:
                self._cache[key] = ops.anchors_pyramid(feature_hws, image_hw, device, self.sizes, self.aspect_ratios)
            return self._cache[key]

    _default_anchors = None

    @staticmethod
    def region_proposal(cls, reg, anchor=None, mode="train", image_hw=None, feature_hws=None):
        """Proposal part of ``RegionProposalNetwork.forward`` (models/new_model.py:46-83): cls [N,2] logits and reg [N,4]
        of all pyramid levels concatenated -> rois [<=1000, 4].  ``anchor`` [N,4] normalised, or None: the reference's
        5-level torchvision anchors are generated on the device from ``image_hw`` and the pyramid's ``feature_hws``.
        Same kernels as the VGG variant with min_size 10/1000 and 4000|2000 -> 1000."""
        pre_k, post_k = fpn.PROPOSAL_MODES["test" if mode == "test" else "train"]
        if anchor is None:
            if image_hw is None or feature_hws is None:
                raise ValueError("region_proposal: give the anchors, or image_hw and feature_hws to generate them")
            if fpn._default_anchors is None:
                fpn._default_anchors = fpn.AnchorGenerator()
            anchor = fpn._default_anchors(image_hw, feature_hws, reg.device)
        anchor = _as_anchor_tensor(anchor, reg.device)
        rois, count = region.rpn_proposals(cls.detach().unsqueeze(0).to(torch.float32),
                                           reg.detach().unsqueeze(0).to(torch.float32), anchors=anchor, mode="train",
                                           pre_nms_top_k=pre_k, post_nms_top_k=post_k, min_size=fpn.MIN_SIZE)
        return rois[0, :int(count[0])]

    class RPNTargetMaker(nn.Module):
        """models/new_model.py:299-349.  ``forward(boxes [G,4], anchors [N,4])`` -> (label int64 [N], tg_cxywh [N,4])."""

        def forward(self, boxes, anchors):
            anchors = _as_anchor_tensor(anchors, boxes.device)
            labels, reg = targets.rpn_targets(boxes.detach().to(torch.float32).reshape(1, -1, 4), None, anchors=anchors,
                                              variant="fpn")
            return labels[0], reg[0]

    class FRCNNTargetMaker(nn.Module):
        """models/new_model.py:153-206.  ``forward(boxes [G,4], labels [G], rois [R,4])`` ->
        (cls int64 [<=512], reg [<=512,4], sample_rois [<=512,4])."""

        def forward(self, boxes, labels, rois):
            cls, reg, srois, _, n = targets.frcnn_targets(rois.detach().to(torch.float32).unsqueeze(0), None,
                                                          boxes.detach().to(torch.float32).unsqueeze(0), None,
                                                          labels.detach().to(torch.int64).unsqueeze(0), variant="fpn")
            k = int(n[0])
            return cls[0, :k], reg[0, :k], srois[0, :k]


class RPNLoss(nn.Module):
    """Drop-in for losses/loss.py:17-41: ``forward(pred_cls [1,N,2], pred_reg [1,N,4], target_cls [N], target_reg [N,4])``
    -> (rpn_cls_loss, rpn_reg_loss), differentiable w.r.t. the predictions (one fused kernel)."""

    def forward(self, pred_cls, pred_reg, target_cls, target_reg):
        n = target_cls.shape[-1]
        loss = ops.region_loss(rpn_cls=pred_cls.reshape(1, n, 2), rpn_reg=pred_reg.reshape(1, n, 4),
                               rpn_target_cls=target_cls.reshape(1, n).to(torch.int64),
                               rpn_target_reg=target_reg.reshape(1, n, 4))
        return loss[0, 1], loss[0, 2]


class FastRCNNLoss(nn.Module):
    """Drop-in for losses/loss.py:44-59: ``forward(pred_cls [S,C], pred_reg, target_cls [S], target_reg [S,4])`` ->
    (fast_rcnn_cls_loss, fast_rcnn_reg_loss).  ``pred_reg`` is either the gathered [S,4] the reference passes
    (models/model.py:340-341) or the head's [S,C*4]: the class row is then picked inside the kernel."""

    def forward(self, pred_cls, pred_reg, target_cls, target_reg):
        s = target_cls.shape[-1]
        c = pred_cls.shape[-1]
        loss = ops.region_loss(frcnn_cls=pred_cls.reshape(1, s, c), frcnn_reg=pred_reg.reshape(1, s, -1),
                               frcnn_target_cls=target_cls.reshape(1, s).to(torch.int64),
                               frcnn_target_reg=target_reg.reshape(1, s, 4))
        return loss[0, 3], loss[0, 4]


class FRCNNLoss(nn.Module):
    """Drop-in for losses/loss.py:62-82: ``forward(pred, target)`` with the 4-tuples of ``FRCNN.forward`` ->
    (total, rpn_cls, rpn_reg, fast_rcnn_cls, fast_rcnn_reg)."""

    def __init__(self, opts=None):
        super().__init__()
        self.opts = opts

    def forward(self, pred, target):
        rc, rr, fc, fr = pred
        t_rc, t_rr, t_fc, t_fr = target
        n, s, c = t_rc.shape[-1], t_fc.shape[-1], fc.shape[-1]
        loss = ops.region_loss(rc.reshape(1, n, 2), rr.reshape(1, n, 4), t_rc.reshape(1, n).to(torch.int64),
                               t_rr.reshape(1, n, 4), fc.reshape(1, s, c), fr.reshape(1, s, -1),
                               t_fc.reshape(1, s).to(torch.int64), t_fr.reshape(1, s, 4))
        return loss[0, 0], loss[0, 1], loss[0, 2], loss[0, 3], loss[0, 4]


def predict_tail(pred_cls, pred_reg, rois, num_classes: int):
    """models/model.py:369-378: (prob [R,C], clamped per-class boxes [R,4C])."""
    return ops.decode_classwise(pred_cls.detach().to(torch.float32), pred_reg.detach().to(torch.float32).reshape(-1, num_classes * 4),
                                rois.detach().to(torch.float32), num_classes)


def suppress(raw_cls_bbox, raw_prob, num_classes: int, thres: float):
    """``FRCNN._suppress`` (models/model.py:382-402): numpy (bbox f32 [D,4], label i32 [D], score f32 [D])."""
    R = raw_prob.shape[0]
    db, dl, ds, dc = ops.class_nms(raw_prob.detach().to(torch.float32).reshape(1, R, num_classes),
                                   raw_cls_bbox.detach().to(torch.float32).reshape(1, R, num_classes * 4), num_classes,
                                   score_thres=thres, iou_thr=0.3)
    d = int(dc[0])                        # one host sync (the reference: two per class)
    return (db[0, :d].cpu().numpy().astype(np.float32), dl[0, :d].cpu().numpy().astype(np.int32),
            ds[0, :d].cpu().numpy().astype(np.float32))
