"""``torch.ops.frr.*``: the region-stage kernels registered as PyTorch custom ops (``torch.library.custom_op`` with fake
/ meta implementations and autograd formulas), with the schemas of the torchvision ops the reference calls
(SURVEY 8b; models/model.py:6-9,53,97,113,394; models/new_model.py:127,143):

    frr::nms(Tensor dets, Tensor scores, float iou_threshold) -> Tensor
    frr::roi_pool(Tensor input, Tensor rois, float spatial_scale, SymInt pooled_height, SymInt pooled_width) -> (Tensor, Tensor)
    frr::_roi_pool_backward(Tensor grad, Tensor rois, Tensor argmax, float spatial_scale, SymInt pooled_height,
                            SymInt pooled_width, SymInt batch_size, SymInt channels, SymInt height, SymInt width) -> Tensor
    frr::roi_align(Tensor input, Tensor rois, float spatial_scale, SymInt pooled_height, SymInt pooled_width,
                   int sampling_ratio, bool aligned) -> Tensor
    frr::_roi_align_backward(Tensor grad, Tensor rois, float spatial_scale, SymInt pooled_height, SymInt pooled_width,
                             SymInt batch_size, SymInt channels, SymInt height, SymInt width, int sampling_ratio,
                             bool aligned) -> Tensor
    frr::rpn_proposals(Tensor cls, Tensor reg, int image_h, int image_w, int pre_nms_top_k, int post_nms_top_k,
                       float nms_thresh, float min_size) -> (Tensor rois, Tensor count)

and the rest of the batched region stage (``region`` / ``targets`` / ``ops``), so that whole predict and train steps
compile with ``torch.compile(fullgraph=True)`` (``int`` arguments are ``SymInt`` in the registered schemas):

    frr::rpn_proposals_sized(Tensor cls, Tensor reg, Tensor image_hw, int grid_h, int grid_w, int pre_nms_top_k,
                             int post_nms_top_k, float nms_thresh, float min_size) -> (Tensor rois, Tensor count)
    frr::rpn_proposals_anchored(Tensor cls, Tensor reg, Tensor anchors, int pre_nms_top_k, int post_nms_top_k,
                                float nms_thresh, float min_size) -> (Tensor rois, Tensor count)
    frr::rois5(Tensor rois, Tensor? count, int feat_h, int feat_w, Tensor? image_hw, int stride) -> Tensor
    frr::roi_pool_sized(Tensor input, Tensor rois, Tensor image_hw, float spatial_scale, int pooled_height,
                        int pooled_width, int stride) -> (Tensor, Tensor)
    frr::_roi_pool_backward_sized(Tensor grad, Tensor rois, Tensor argmax, Tensor image_hw, float spatial_scale,
                                  int pooled_height, int pooled_width, int batch_size, int channels, int height, int width,
                                  int stride) -> Tensor
    frr::make_targets(Tensor gt, Tensor? gt_count, Tensor gt_label, Tensor rois, Tensor? roi_count, Tensor(a!) mt_state,
                      int image_h, int image_w, Tensor? image_hw)
        -> (rpn_cls, rpn_reg, frcnn_cls, frcnn_reg, sample_rois, keep_index, n_samples)
    frr::rpn_targets(Tensor gt, Tensor? gt_count, Tensor(a!) mt_state, Tensor? anchors, int image_h, int image_w,
                     Tensor? image_hw, str variant) -> (Tensor labels, Tensor reg)
    frr::frcnn_targets(Tensor rois, Tensor? roi_count, Tensor gt, Tensor? gt_count, Tensor gt_label, Tensor(a!) mt_state,
                       str variant) -> (cls, reg, sample_rois, keep_index, n_samples)
    frr::region_loss(Tensor? rpn_cls, Tensor? rpn_reg, Tensor? rpn_target_cls, Tensor? rpn_target_reg,
                     Tensor? frcnn_cls, Tensor? frcnn_reg, Tensor? frcnn_target_cls, Tensor? frcnn_target_reg)
        -> (loss [B,5], grad_rpn_cls, grad_rpn_reg, grad_frcnn_cls, grad_frcnn_reg)
    frr::decode_classwise(Tensor cls_logits, Tensor reg, Tensor rois, int num_classes) -> (Tensor prob, Tensor boxes)
    frr::class_nms(Tensor prob, Tensor boxes, int num_classes, float score_thres, float iou_thr, Tensor? roi_count,
                   int? cap) -> (det_boxes, det_labels, det_scores, det_count)
    frr::pack_detections(Tensor det_boxes, Tensor det_labels, Tensor det_scores, Tensor det_count, int max_det,
                         Tensor? image_wh, bool xywh, str rank, int per_class_max) -> (Tensor rows, Tensor count)
    frr::multiscale_roi_align(Tensor[] features, Tensor rois, int pooled_height, int pooled_width, int sampling_ratio,
                              float[] scales, int k_min, int k_max, float canonical_scale, int canonical_level)
        -> (Tensor out, Tensor levels, Tensor level_rois)
    frr::_multiscale_roi_align_backward(Tensor grad, Tensor level_rois, int[] feature_shapes, float[] scales,
                                        int sampling_ratio) -> Tensor[]

Importing this module registers the ops; every implementation is a libfrr kernel (CUDA tensors only, no CPU kernel is
registered: a CPU call fails in the dispatcher).  The fake implementations make the ops traceable (``torch.compile`` /
``make_fx`` / meta tensors) with the right output shapes; ``nms`` has a data-dependent output length (unbacked SymInt).
Autograd formulas: ``roi_pool``, ``roi_align``, ``roi_pool_sized`` and ``multiscale_roi_align`` (one gradient per
level) w.r.t. the features; ``region_loss`` w.r.t. its four predictions (its extra outputs are the kernel's gradients
for a unit upstream gradient, which the backward scales).  The RoI backward ops read ``torch.use_deterministic_algorithms``
when they run; a captured CUDA graph keeps the kernel chosen at capture.  The target ops sample on the device from
``mt_state`` (``targets.DeviceGenerator.state``, the only argument any op mutates): no op synchronises with the host,
and host-sampled targets have no op.
"""
from __future__ import annotations

import torch

from . import ops, region, targets

_LIB = "frr"


@torch.library.custom_op(f"{_LIB}::nms", mutates_args=(), device_types="cuda")
def nms(dets: torch.Tensor, scores: torch.Tensor, iou_threshold: float) -> torch.Tensor:
    from .modules import nms as _nms
    return _nms(dets, scores, iou_threshold)


@nms.register_fake
def _(dets, scores, iou_threshold):
    n = torch.library.get_ctx().new_dynamic_size()
    return dets.new_empty((n,), dtype=torch.int64)


@torch.library.custom_op(f"{_LIB}::roi_pool", mutates_args=(), device_types="cuda")
def roi_pool(input: torch.Tensor, rois: torch.Tensor, spatial_scale: float, pooled_height: int,
             pooled_width: int) -> tuple[torch.Tensor, torch.Tensor]:
    feat, _ = ops._feat_layout(input)
    return ops.roi_pool_forward(feat, rois.to(torch.float32).contiguous(), (pooled_height, pooled_width), spatial_scale, True)


@roi_pool.register_fake
def _(input, rois, spatial_scale, pooled_height, pooled_width):
    shape = (rois.shape[0], input.shape[1], pooled_height, pooled_width)
    return input.new_empty(shape), input.new_empty(shape, dtype=torch.int32)


@torch.library.custom_op(f"{_LIB}::_roi_pool_backward", mutates_args=(), device_types="cuda")
def _roi_pool_backward(grad: torch.Tensor, rois: torch.Tensor, argmax: torch.Tensor, spatial_scale: float, pooled_height: int,
                       pooled_width: int, batch_size: int, channels: int, height: int, width: int) -> torch.Tensor:
    return ops.roi_pool_backward(grad.contiguous(), argmax, rois.to(torch.float32).contiguous(),
                                 (batch_size, channels, height, width), spatial_scale, False)


@_roi_pool_backward.register_fake
def _(grad, rois, argmax, spatial_scale, pooled_height, pooled_width, batch_size, channels, height, width):
    return grad.new_empty((batch_size, channels, height, width))


def _roi_pool_setup(ctx, inputs, output):
    input, rois, spatial_scale, ph, pw = inputs
    ctx.save_for_backward(rois, output[1])
    ctx.meta = (spatial_scale, ph, pw, tuple(input.shape))
    ctx.mark_non_differentiable(output[1])


def _roi_pool_bwd(ctx, grad_out, _grad_argmax):
    rois, argmax = ctx.saved_tensors
    scale, ph, pw, (b, c, h, w) = ctx.meta
    return torch.ops.frr._roi_pool_backward(grad_out, rois, argmax, scale, ph, pw, b, c, h, w), None, None, None, None


torch.library.register_autograd(f"{_LIB}::roi_pool", _roi_pool_bwd, setup_context=_roi_pool_setup)


@torch.library.custom_op(f"{_LIB}::roi_align", mutates_args=(), device_types="cuda")
def roi_align(input: torch.Tensor, rois: torch.Tensor, spatial_scale: float, pooled_height: int, pooled_width: int,
              sampling_ratio: int, aligned: bool) -> torch.Tensor:
    feat, _ = ops._feat_layout(input)
    return ops.roi_align_forward(feat, rois.to(torch.float32).contiguous(), (pooled_height, pooled_width), spatial_scale,
                                 sampling_ratio, aligned)


@roi_align.register_fake
def _(input, rois, spatial_scale, pooled_height, pooled_width, sampling_ratio, aligned):
    return input.new_empty((rois.shape[0], input.shape[1], pooled_height, pooled_width))


@torch.library.custom_op(f"{_LIB}::_roi_align_backward", mutates_args=(), device_types="cuda")
def _roi_align_backward(grad: torch.Tensor, rois: torch.Tensor, spatial_scale: float, pooled_height: int, pooled_width: int,
                        batch_size: int, channels: int, height: int, width: int, sampling_ratio: int,
                        aligned: bool) -> torch.Tensor:
    return ops.roi_align_backward(grad.contiguous(), rois.to(torch.float32).contiguous(), (batch_size, channels, height, width),
                                  spatial_scale, sampling_ratio, aligned, False)


@_roi_align_backward.register_fake
def _(grad, rois, spatial_scale, pooled_height, pooled_width, batch_size, channels, height, width, sampling_ratio, aligned):
    return grad.new_empty((batch_size, channels, height, width))


def _roi_align_setup(ctx, inputs, output):
    input, rois, spatial_scale, ph, pw, sampling_ratio, aligned = inputs
    ctx.save_for_backward(rois)
    ctx.meta = (spatial_scale, ph, pw, sampling_ratio, aligned, tuple(input.shape))


def _roi_align_bwd(ctx, grad_out):
    (rois,) = ctx.saved_tensors
    scale, ph, pw, sr, aligned, (b, c, h, w) = ctx.meta
    return (torch.ops.frr._roi_align_backward(grad_out, rois, scale, ph, pw, b, c, h, w, sr, aligned),
            None, None, None, None, None, None)


torch.library.register_autograd(f"{_LIB}::roi_align", _roi_align_bwd, setup_context=_roi_align_setup)


@torch.library.custom_op(f"{_LIB}::rpn_proposals", mutates_args=(), device_types="cuda")
def rpn_proposals(cls: torch.Tensor, reg: torch.Tensor, image_h: int, image_w: int, pre_nms_top_k: int, post_nms_top_k: int,
                  nms_thresh: float, min_size: float) -> tuple[torch.Tensor, torch.Tensor]:
    """Batched RegionProposal.forward (models/model.py:17-58): cls [B,N,2] logits or [B,N] scores, reg [B,N,4] ->
    rois [B,post,4] (zero padded), count int32 [B]."""
    rois, count = region.rpn_proposals(cls, reg, image_hw=(image_h, image_w), pre_nms_top_k=pre_nms_top_k,
                                       post_nms_top_k=post_nms_top_k, nms_thresh=nms_thresh, min_size=min_size)
    return rois, count


@rpn_proposals.register_fake
def _(cls, reg, image_h, image_w, pre_nms_top_k, post_nms_top_k, nms_thresh, min_size):
    return reg.new_empty((reg.shape[0], post_nms_top_k, 4)), reg.new_empty((reg.shape[0],), dtype=torch.int32)


# ------------------------------------------------------------------------------------------------
# the batched region stage: mixed-size and FPN proposals, rois, targets, loss, detection tail, MultiScaleRoIAlign
# ------------------------------------------------------------------------------------------------
def _empty(like, *shape, dtype=torch.float32):
    return like.new_empty(shape, dtype=dtype)


@torch.library.custom_op(f"{_LIB}::rpn_proposals_sized", mutates_args=(), device_types="cuda")
def rpn_proposals_sized(cls: torch.Tensor, reg: torch.Tensor, image_hw: torch.Tensor, grid_h: int, grid_w: int,
                        pre_nms_top_k: int, post_nms_top_k: int, nms_thresh: float,
                        min_size: float) -> tuple[torch.Tensor, torch.Tensor]:
    """Mixed-size batch: ``image_hw`` int32 [B,2] per-image (H, W) on the device, N = grid_h * grid_w * 9."""
    return region.rpn_proposals(cls, reg, image_hw=image_hw, grid_hw=(grid_h, grid_w), pre_nms_top_k=pre_nms_top_k,
                                post_nms_top_k=post_nms_top_k, nms_thresh=nms_thresh, min_size=min_size)


@torch.library.custom_op(f"{_LIB}::rpn_proposals_anchored", mutates_args=(), device_types="cuda")
def rpn_proposals_anchored(cls: torch.Tensor, reg: torch.Tensor, anchors: torch.Tensor, pre_nms_top_k: int,
                           post_nms_top_k: int, nms_thresh: float, min_size: float) -> tuple[torch.Tensor, torch.Tensor]:
    """Given normalised anchors [N,4] (the FPN variant: ``ops.anchors_pyramid``)."""
    return region.rpn_proposals(cls, reg, anchors=anchors, pre_nms_top_k=pre_nms_top_k, post_nms_top_k=post_nms_top_k,
                                nms_thresh=nms_thresh, min_size=min_size)


@rpn_proposals_sized.register_fake
def _(cls, reg, image_hw, grid_h, grid_w, pre_nms_top_k, post_nms_top_k, nms_thresh, min_size):
    return _empty(reg, reg.shape[0], post_nms_top_k, 4), _empty(reg, reg.shape[0], dtype=torch.int32)


@rpn_proposals_anchored.register_fake
def _(cls, reg, anchors, pre_nms_top_k, post_nms_top_k, nms_thresh, min_size):
    return _empty(reg, reg.shape[0], post_nms_top_k, 4), _empty(reg, reg.shape[0], dtype=torch.int32)


@torch.library.custom_op(f"{_LIB}::rois5", mutates_args=(), device_types="cuda")
def rois5(rois: torch.Tensor, count: torch.Tensor | None, feat_h: int, feat_w: int, image_hw: torch.Tensor | None,
          stride: int) -> torch.Tensor:
    return ops.rois5(rois, count, (feat_h, feat_w), image_hw=image_hw, stride=stride)


@rois5.register_fake
def _(rois, count, feat_h, feat_w, image_hw, stride):
    return _empty(rois, rois.shape[0] * rois.shape[1], 5)


@torch.library.custom_op(f"{_LIB}::roi_pool_sized", mutates_args=(), device_types="cuda")
def roi_pool_sized(input: torch.Tensor, rois: torch.Tensor, image_hw: torch.Tensor, spatial_scale: float, pooled_height: int,
                   pooled_width: int, stride: int) -> tuple[torch.Tensor, torch.Tensor]:
    """``roi_pool`` of a mixed-size batch: bin windows of image b clipped to its grid (H_b // stride, W_b // stride)."""
    feat, _ = ops._feat_layout(input)
    return ops.roi_pool_forward(feat, rois.to(torch.float32).contiguous(), (pooled_height, pooled_width), spatial_scale, True,
                                image_hw=image_hw, stride=stride)


@roi_pool_sized.register_fake
def _(input, rois, image_hw, spatial_scale, pooled_height, pooled_width, stride):
    shape = (rois.shape[0], input.shape[1], pooled_height, pooled_width)
    return input.new_empty(shape), input.new_empty(shape, dtype=torch.int32)


@torch.library.custom_op(f"{_LIB}::_roi_pool_backward_sized", mutates_args=(), device_types="cuda")
def _roi_pool_backward_sized(grad: torch.Tensor, rois: torch.Tensor, argmax: torch.Tensor, image_hw: torch.Tensor,
                             spatial_scale: float, pooled_height: int, pooled_width: int, batch_size: int, channels: int,
                             height: int, width: int, stride: int) -> torch.Tensor:
    return ops.roi_pool_backward(grad.contiguous(), argmax, rois.to(torch.float32).contiguous(),
                                 (batch_size, channels, height, width), spatial_scale, False, image_hw=image_hw, stride=stride)


@_roi_pool_backward_sized.register_fake
def _(grad, rois, argmax, image_hw, spatial_scale, pooled_height, pooled_width, batch_size, channels, height, width, stride):
    return grad.new_empty((batch_size, channels, height, width))


def _roi_pool_sized_setup(ctx, inputs, output):
    input, rois, image_hw, spatial_scale, ph, pw, stride = inputs
    ctx.save_for_backward(rois, output[1], image_hw)
    ctx.meta = (spatial_scale, ph, pw, tuple(input.shape), stride)
    ctx.mark_non_differentiable(output[1])


def _roi_pool_sized_bwd(ctx, grad_out, _grad_argmax):
    rois, argmax, image_hw = ctx.saved_tensors
    scale, ph, pw, (b, c, h, w), stride = ctx.meta
    return (torch.ops.frr._roi_pool_backward_sized(grad_out, rois, argmax, image_hw, scale, ph, pw, b, c, h, w, stride),
            None, None, None, None, None, None)


torch.library.register_autograd(f"{_LIB}::roi_pool_sized", _roi_pool_sized_bwd, setup_context=_roi_pool_sized_setup)


class _Generator:
    """what ``targets.*`` reads of a ``DeviceGenerator``: its device-resident mt19937 state"""

    def __init__(self, state):
        self.state = state


def _grid(image_h, image_w, stride=16):
    return image_h // stride, image_w // stride


@torch.library.custom_op(f"{_LIB}::make_targets", mutates_args=("mt_state",), device_types="cuda")
def make_targets(gt: torch.Tensor, gt_count: torch.Tensor | None, gt_label: torch.Tensor, rois: torch.Tensor,
                 roi_count: torch.Tensor | None, mt_state: torch.Tensor, image_h: int, image_w: int,
                 image_hw: torch.Tensor | None) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor,
                                                         torch.Tensor, torch.Tensor]:
    """``targets.make_targets`` with device sampling from ``mt_state`` (``DeviceGenerator.state``, advanced in place).
    (image_h, image_w): the batch's (padded) size, grid (image_h // 16, image_w // 16); ``image_hw`` int32 [B,2]: the
    per-image sizes of a mixed-size batch.  Returns (rpn_cls, rpn_reg, frcnn_cls, frcnn_reg, sample_rois, keep_index,
    n_samples)."""
    t = targets.make_targets(gt, gt_count, gt_label, rois, roi_count,
                             image_hw=(image_h, image_w) if image_hw is None else image_hw, generator=_Generator(mt_state),
                             grid_hw=_grid(image_h, image_w))
    return (t["rpn_cls"], t["rpn_reg"], t["frcnn_cls"], t["frcnn_reg"], t["sample_rois"], t["keep_index"],
            t["n_samples"].contiguous())


@make_targets.register_fake
def _(gt, gt_count, gt_label, rois, roi_count, mt_state, image_h, image_w, image_hw):
    B, S = gt.shape[0], targets.FRCNN_BATCH
    gh, gw = _grid(image_h, image_w)
    N = gh * gw * 9
    return (_empty(gt, B, N, dtype=torch.int64), _empty(gt, B, N, 4), _empty(gt, B, S, dtype=torch.int64),
            _empty(gt, B, S, 4), _empty(gt, B, S, 4), _empty(gt, B, S, dtype=torch.int32), _empty(gt, B, dtype=torch.int32))


@torch.library.custom_op(f"{_LIB}::rpn_targets", mutates_args=("mt_state",), device_types="cuda")
def rpn_targets(gt: torch.Tensor, gt_count: torch.Tensor | None, mt_state: torch.Tensor, anchors: torch.Tensor | None,
                image_h: int, image_w: int, image_hw: torch.Tensor | None, variant: str) -> tuple[torch.Tensor, torch.Tensor]:
    """``targets.rpn_targets`` with device sampling: labels int64 [B,N], reg [B,N,4].  ``anchors`` [N,4] (FPN) or
    anchors generated for (image_h, image_w) (+ per-image ``image_hw``, as in ``make_targets``)."""
    if anchors is not None:
        return targets.rpn_targets(gt, gt_count, anchors=anchors, generator=_Generator(mt_state), variant=variant)
    return targets.rpn_targets(gt, gt_count, image_hw=(image_h, image_w) if image_hw is None else image_hw,
                               generator=_Generator(mt_state), grid_hw=_grid(image_h, image_w), variant=variant)


@rpn_targets.register_fake
def _(gt, gt_count, mt_state, anchors, image_h, image_w, image_hw, variant):
    gh, gw = _grid(image_h, image_w)
    N = anchors.shape[0] if anchors is not None else gh * gw * 9
    return _empty(gt, gt.shape[0], N, dtype=torch.int64), _empty(gt, gt.shape[0], N, 4)


@torch.library.custom_op(f"{_LIB}::frcnn_targets", mutates_args=("mt_state",), device_types="cuda")
def frcnn_targets(rois: torch.Tensor, roi_count: torch.Tensor | None, gt: torch.Tensor, gt_count: torch.Tensor | None,
                  gt_label: torch.Tensor, mt_state: torch.Tensor,
                  variant: str) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """``targets.frcnn_targets`` with device sampling: (cls, reg, sample_rois, keep_index, n_samples), S = 128 ("vgg")
    or 512 ("fpn") samples per image."""
    cls, reg, srois, kidx, n = targets.frcnn_targets(rois, roi_count, gt, gt_count, gt_label, variant=variant,
                                                     generator=_Generator(mt_state))
    return cls, reg, srois, kidx, n.contiguous()


@frcnn_targets.register_fake
def _(rois, roi_count, gt, gt_count, gt_label, mt_state, variant):
    B, S = rois.shape[0], targets.FRCNN_SAMPLING[variant][0]
    return (_empty(rois, B, S, dtype=torch.int64), _empty(rois, B, S, 4), _empty(rois, B, S, 4),
            _empty(rois, B, S, dtype=torch.int32), _empty(rois, B, dtype=torch.int32))


@torch.library.custom_op(f"{_LIB}::region_loss", mutates_args=(), device_types="cuda")
def region_loss(rpn_cls: torch.Tensor | None, rpn_reg: torch.Tensor | None, rpn_target_cls: torch.Tensor | None,
                rpn_target_reg: torch.Tensor | None, frcnn_cls: torch.Tensor | None, frcnn_reg: torch.Tensor | None,
                frcnn_target_cls: torch.Tensor | None, frcnn_target_reg: torch.Tensor | None
                ) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """``ops.region_loss``: loss [B,5], then the kernel's gradients of each image's total w.r.t. rpn_cls, rpn_reg,
    frcnn_cls, frcnn_reg (shaped like them; an empty tensor for an omitted half).  Only the loss is differentiable; its
    backward scales the four saved gradients."""
    args = ops.region_loss_args(rpn_cls, rpn_reg, rpn_target_cls, rpn_target_reg, frcnn_cls, frcnn_reg, frcnn_target_cls,
                                frcnn_target_reg)
    loss, grads = ops.region_loss_kernel(*args, need=(True,) * 4)
    preds = (rpn_cls, rpn_reg, frcnn_cls, frcnn_reg)
    return (loss,) + tuple(loss.new_empty((0,)) if g is None else g.view(p.shape) for g, p in zip(grads, preds))


@region_loss.register_fake
def _(rpn_cls, rpn_reg, rpn_target_cls, rpn_target_reg, frcnn_cls, frcnn_reg, frcnn_target_cls, frcnn_target_reg):
    ref = rpn_cls if rpn_cls is not None else frcnn_cls
    return (_empty(ref, ref.shape[0], 5),) + tuple(_empty(ref, 0) if p is None else p.new_empty(p.shape)
                                                   for p in (rpn_cls, rpn_reg, frcnn_cls, frcnn_reg))


def _region_loss_setup(ctx, inputs, output):
    ctx.have = tuple(inputs[j] is not None for j in (0, 1, 4, 5))
    ctx.save_for_backward(*output[1:])
    ctx.mark_non_differentiable(*output[1:])


def _region_loss_bwd(ctx, g, *_grad_saved):
    saved = [s if h else None for s, h in zip(ctx.saved_tensors, ctx.have)]
    g_rc, g_rr, g_fc, g_fr = ops.region_loss_scale(saved, g)
    return g_rc, g_rr, None, None, g_fc, g_fr, None, None


torch.library.register_autograd(f"{_LIB}::region_loss", _region_loss_bwd, setup_context=_region_loss_setup)


@torch.library.custom_op(f"{_LIB}::decode_classwise", mutates_args=(), device_types="cuda")
def decode_classwise(cls_logits: torch.Tensor, reg: torch.Tensor, rois: torch.Tensor,
                     num_classes: int) -> tuple[torch.Tensor, torch.Tensor]:
    return ops.decode_classwise(cls_logits, reg, rois, num_classes)


@decode_classwise.register_fake
def _(cls_logits, reg, rois, num_classes):
    rows = cls_logits.shape[0]
    return _empty(cls_logits, rows, num_classes), _empty(cls_logits, rows, 4 * num_classes)


@torch.library.custom_op(f"{_LIB}::class_nms", mutates_args=(), device_types="cuda")
def class_nms(prob: torch.Tensor, boxes: torch.Tensor, num_classes: int, score_thres: float, iou_thr: float,
              roi_count: torch.Tensor | None, cap: int | None) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    return ops.class_nms(prob, boxes, num_classes, score_thres, iou_thr, roi_count=roi_count, cap=cap)


@class_nms.register_fake
def _(prob, boxes, num_classes, score_thres, iou_thr, roi_count, cap):
    B, R = prob.shape[0], prob.shape[1]
    cap = R * (num_classes - 1) if cap is None else cap
    return (_empty(prob, B, cap, 4), _empty(prob, B, cap, dtype=torch.int32), _empty(prob, B, cap),
            _empty(prob, B, dtype=torch.int32))


@torch.library.custom_op(f"{_LIB}::pack_detections", mutates_args=(), device_types="cuda")
def pack_detections(det_boxes: torch.Tensor, det_labels: torch.Tensor, det_scores: torch.Tensor, det_count: torch.Tensor,
                    max_det: int, image_wh: torch.Tensor | None, xywh: bool, rank: str,
                    per_class_max: int) -> tuple[torch.Tensor, torch.Tensor]:
    """``ops.pack_detections``; the ranking workspace of ``rank="score"`` is allocated by each call."""
    return ops.pack_detections(det_boxes, det_labels, det_scores, det_count, max_det, image_wh=image_wh, xywh=xywh, rank=rank,
                               per_class_max=per_class_max)


@pack_detections.register_fake
def _(det_boxes, det_labels, det_scores, det_count, max_det, image_wh, xywh, rank, per_class_max):
    ops.check_rank(rank, per_class_max)
    B = det_labels.shape[0]
    return _empty(det_boxes, B, max_det, 6), _empty(det_boxes, B, dtype=torch.int32)


@torch.library.custom_op(f"{_LIB}::multiscale_roi_align", mutates_args=(), device_types="cuda")
def multiscale_roi_align(features: list[torch.Tensor], rois: torch.Tensor, pooled_height: int, pooled_width: int,
                         sampling_ratio: int, scales: list[float], k_min: int, k_max: int, canonical_scale: float,
                         canonical_level: int) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """``ops.multiscale_roi_align`` of [K,5] image-coordinate rois over the levels k_min..k_max (one feature map and one
    scale per level, ``ops.infer_scales``): (out [K,C,PH,PW], levels int32 [K], per-level rois [L,K,5] for the
    backward)."""
    if len(features) != k_max - k_min + 1 or len(scales) != len(features):
        raise ValueError("multiscale_roi_align: one feature map and one scale per level k_min..k_max")
    out, levels, per, _ = ops.multiscale_roi_align_forward(features, rois.to(torch.float32).contiguous(),
                                                           (pooled_height, pooled_width), sampling_ratio, scales, k_min,
                                                           k_max, canonical_scale, canonical_level)
    return out, levels, per


@multiscale_roi_align.register_fake
def _(features, rois, pooled_height, pooled_width, sampling_ratio, scales, k_min, k_max, canonical_scale, canonical_level):
    K = rois.shape[0]
    return (_empty(rois, K, features[0].shape[1], pooled_height, pooled_width), _empty(rois, K, dtype=torch.int32),
            _empty(rois, k_max - k_min + 1, K, 5))


@torch.library.custom_op(f"{_LIB}::_multiscale_roi_align_backward", mutates_args=(), device_types="cuda")
def _multiscale_roi_align_backward(grad: torch.Tensor, level_rois: torch.Tensor, feature_shapes: list[int],
                                   scales: list[float], sampling_ratio: int) -> list[torch.Tensor]:
    """One NCHW-contiguous gradient per level; ``feature_shapes``: (B, C, H, W) of every level, concatenated."""
    shapes = [tuple(feature_shapes[4 * l:4 * l + 4]) for l in range(len(scales))]
    return ops.multiscale_roi_align_backward(grad, level_rois, shapes, scales, sampling_ratio, [False] * len(scales))


@_multiscale_roi_align_backward.register_fake
def _(grad, level_rois, feature_shapes, scales, sampling_ratio):
    return [grad.new_empty(tuple(feature_shapes[4 * l:4 * l + 4])) for l in range(len(scales))]


def _msroi_setup(ctx, inputs, output):
    features, _, _, _, sampling_ratio, scales, *_ = inputs
    ctx.save_for_backward(output[2])
    ctx.meta = ([d for f in features for d in f.shape], list(scales), sampling_ratio)
    ctx.mark_non_differentiable(output[1], output[2])


def _msroi_bwd(ctx, grad_out, _grad_levels, _grad_level_rois):
    (per,) = ctx.saved_tensors
    shapes, scales, sr = ctx.meta
    return (torch.ops.frr._multiscale_roi_align_backward(grad_out, per, shapes, scales, sr),) + (None,) * 9


torch.library.register_autograd(f"{_LIB}::multiscale_roi_align", _msroi_bwd, setup_context=_msroi_setup)
