"""Tensor-level wrappers over the C ABI (include/frr.h).

PyTorch is plumbing here: it owns device memory and streams; every computation is a kernel of
libfrr.so.  All functions require CUDA fp32 tensors and raise otherwise (no CPU fallback).
Batched layouts: a leading ``B`` dimension = images; ragged results come back as
fixed-capacity tensors + ``int32 count[B]`` on the device (no host sync).
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib

_MIN_SIZE = float(np.float32(1.0 / 1000.0))  # models/model.py:39, compared in fp32


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _req(t: torch.Tensor, name: str, dtype=torch.float32):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor: the region stage has no CPU path")
    if t.dtype != dtype:
        raise ValueError(f"{name} must be {dtype}, got {t.dtype}")
    return t.contiguous()


def anchor_base_table(base_size: int = 16) -> np.ndarray:
    """anchor.py:15-32 (host, 9x4 fp32)."""
    out = np.empty((9, 4), dtype=np.float32)
    _lib.check(_lib.load().frr_anchor_base_host(out.ctypes.data, int(base_size)), "frr_anchor_base_host")
    return out


def _table_arg(table):
    if table is None:
        return None, 0, 9
    t = np.ascontiguousarray(table, dtype=np.float32).reshape(-1, 4)
    return t, t.ctypes.data, t.shape[0]


def anchors(image_hw, device, stride: int = 16, table=None) -> torch.Tensor:
    """anchor.py:34-55 on the device: [fh*fw*A, 4] fp32, normalised."""
    lib = _lib.load()
    keep, tptr, A = _table_arg(table)
    H, W = int(image_hw[0]), int(image_hw[1])
    n = (H // stride) * (W // stride) * A
    with torch.cuda.device(device):
        out = torch.empty((n, 4), dtype=torch.float32, device=device)
        _lib.check(lib.frr_anchors(out.data_ptr(), H, W, stride, tptr, A, _stream()), "frr_anchors")
    return out


def tv_anchor_base(size: float, aspect_ratios=(0.5, 1.0, 2.0)) -> np.ndarray:
    """torchvision AnchorGenerator.generate_anchors for one level (host, [n_ratios,4] fp32, rounded)."""
    r = np.ascontiguousarray(aspect_ratios, dtype=np.float32)
    out = np.empty((r.shape[0], 4), dtype=np.float32)
    _lib.check(_lib.load().frr_tv_anchor_base_host(float(size), r.ctypes.data, int(r.shape[0]), out.ctypes.data),
               "frr_tv_anchor_base_host")
    return out


def anchors_pyramid(feature_hws, image_hw, device, sizes=(32, 64, 128, 256, 512), aspect_ratios=(0.5, 1.0, 2.0)) -> torch.Tensor:
    """models/new_model.py:43-44 on the device: torchvision's multi-level AnchorGenerator + the division by (w,h,w,h).
    ``feature_hws``: (fh, fw) of every pyramid level; one size per level, the same aspect ratios on every level.
    Returns [sum_l fh_l*fw_l*A, 4] fp32 normalised anchors, levels concatenated."""
    lib = _lib.load()
    L = len(feature_hws)
    if len(sizes) != L:
        raise ValueError("anchors_pyramid: one size per pyramid level")
    tabs = np.stack([tv_anchor_base(float(sz), aspect_ratios) for sz in sizes]).astype(np.float32)      # [L,A,4]
    A = tabs.shape[1]
    hw = np.ascontiguousarray([[int(h), int(w)] for h, w in feature_hws], dtype=np.int32)
    n = int((hw[:, 0] * hw[:, 1]).sum()) * A
    with torch.cuda.device(device):
        out = torch.empty((n, 4), dtype=torch.float32, device=device)
        _lib.check(lib.frr_anchors_pyramid(out.data_ptr(), L, hw.ctypes.data, tabs.ctypes.data, A, int(image_hw[0]),
                                           int(image_hw[1]), _stream()), "frr_anchors_pyramid")
    return out


def rpn_decode(reg, cls, image_hw=None, anchors=None, stride: int = 16, table=None, min_size: float = _MIN_SIZE):
    """Fused A2+P1+P2+P3.  reg [B,N,4]; cls [B,N,2] logits or [B,N] scores.
    Returns boxes [B,N,4], scores [B,N], valid uint8 [B,N]."""
    lib = _lib.load()
    reg = _req(reg, "reg")
    cls = _req(cls, "cls")
    if reg.dim() != 3 or reg.shape[-1] != 4:
        raise ValueError("reg must be [B,N,4]")
    B, N = reg.shape[0], reg.shape[1]
    logits = cls.dim() == 3
    if tuple(cls.shape) != ((B, N, 2) if logits else (B, N)):
        raise ValueError("cls must be [B,N,2] logits or [B,N] scores")
    keep, tptr, A = _table_arg(table)
    if anchors is not None:
        anchors = _req(anchors, "anchors")
        if tuple(anchors.shape) != (N, 4):
            raise ValueError("anchors must be [N,4]")
        H = W = 0
    else:
        if image_hw is None:
            raise ValueError("image_hw is required when anchors are generated in-kernel")
        H, W = int(image_hw[0]), int(image_hw[1])
    with torch.cuda.device(reg.device):
        boxes = torch.empty((B, N, 4), dtype=torch.float32, device=reg.device)
        scores = torch.empty((B, N), dtype=torch.float32, device=reg.device)
        valid = torch.empty((B, N), dtype=torch.uint8, device=reg.device)
        _lib.check(lib.frr_rpn_decode(reg.data_ptr(), cls.data_ptr(), int(logits), _ptr(anchors), tptr, A, H, W, stride,
                                      float(min_size), boxes.data_ptr(), scores.data_ptr(), valid.data_ptr(), B, N,
                                      _stream()), "frr_rpn_decode")
    return boxes, scores, valid


def topk_desc(scores, k: int, valid=None, boxes=None, want_cidx: bool = False, ctas_per_image: int = 0):
    """P4.  scores [B,N] -> dict(scores [B,k], idx int32 [B,k], cidx, boxes [B,k,4], count int32 [B]).
    ``ctas_per_image``: 0 = automatic (a 2-CTA cluster per image for small batches), 1 = one CTA per image."""
    lib = _lib.load()
    scores = _req(scores, "scores")
    if scores.dim() != 2:
        raise ValueError("scores must be [B,N]")
    B, N = scores.shape
    if valid is not None:
        valid = _req(valid, "valid", torch.uint8)
    if boxes is not None:
        boxes = _req(boxes, "boxes")
    dev = scores.device
    with torch.cuda.device(dev):
        o_s = torch.empty((B, k), dtype=torch.float32, device=dev)
        o_i = torch.empty((B, k), dtype=torch.int32, device=dev)
        o_c = torch.empty((B, k), dtype=torch.int32, device=dev) if want_cidx else None
        o_b = torch.empty((B, k, 4), dtype=torch.float32, device=dev) if boxes is not None else None
        cnt = torch.zeros((B,), dtype=torch.int32, device=dev)
        _lib.check(lib.frr_topk_desc_opt(scores.data_ptr(), _ptr(valid), _ptr(boxes), B, N, int(k), o_s.data_ptr(),
                                         o_i.data_ptr(), _ptr(o_c), _ptr(o_b), cnt.data_ptr(), int(ctas_per_image), _stream()),
                   "frr_topk_desc_opt")
    return dict(scores=o_s, idx=o_i, cidx=o_c, boxes=o_b, count=cnt)


def nms_sorted(boxes, iou_threshold: float, max_keep: int | None = None, counts=None, gather: bool = True,
               cluster_size: int = 0, threads: int = 0, dbg=None, unit_boxes: bool = False):
    """N1 on score-sorted boxes [B,n,4].  Returns keep int32 [B,max_keep] (-1 padded), count int32 [B],
    rois [B,max_keep,4] (zero padded) or None.  ``unit_boxes``: the caller guarantees coordinates in [0,1]
    (enables a cheaper, result-identical screening test)."""
    lib = _lib.load()
    boxes = _req(boxes, "boxes")
    if boxes.dim() != 3 or boxes.shape[-1] != 4:
        raise ValueError("boxes must be [B,n,4]")
    B, n = boxes.shape[0], boxes.shape[1]
    mk = n if max_keep is None else int(max_keep)
    if counts is not None:
        counts = _req(counts, "counts", torch.int32)
    dev = boxes.device
    with torch.cuda.device(dev):
        keep = torch.empty((B, mk), dtype=torch.int32, device=dev)
        cnt = torch.empty((B,), dtype=torch.int32, device=dev)
        rois = torch.empty((B, mk, 4), dtype=torch.float32, device=dev) if gather else None
        _lib.check(lib.frr_nms_sorted_tuned(boxes.data_ptr(), _ptr(counts), B, n, float(iou_threshold), mk,
                                            keep.data_ptr(), cnt.data_ptr(), _ptr(rois), int(cluster_size), int(threads),
                                            _ptr(dbg), int(bool(unit_boxes)), _stream()), "frr_nms_sorted")
    return keep, cnt, rois


NMS_VARIANTS = {0: "exact", 1: "screened", 2: "screened+unit", 3: "bucketed"}


def nms_variant(B: int, n: int, iou_threshold: float, max_keep: int | None = None, cluster_size: int = 0,
                threads: int = 0, unit_boxes: bool = False, device=None) -> dict:
    """Kernel variant / launch geometry ``nms_sorted`` picks for this problem (host query, launches nothing)."""
    import ctypes
    out = (ctypes.c_int32 * 4)()
    mk = n if max_keep is None else int(max_keep)
    with torch.cuda.device(device if device is not None else torch.cuda.current_device()):
        _lib.check(_lib.load().frr_nms_variant(int(B), int(n), float(iou_threshold), mk, int(cluster_size), int(threads),
                                               int(bool(unit_boxes)), out), "frr_nms_variant")
    return dict(cluster_size=out[0], threads=out[1], variant=NMS_VARIANTS[out[2]], smem=out[3])


ROI_OPS = {"roi_pool_fwd": 0, "roi_pool_bwd": 1, "roi_align_fwd": 2, "roi_align_bwd": 3}
ROI_KERNELS = {-1: "none", 0: "pool_fwd_flat", 1: "align_fwd_fast", 2: "fwd_planes", 3: "fwd_direct",
               4: "pool_bwd_color_tail", 5: "pool_bwd_tail", 6: "align_bwd_fast", 7: "align_bwd_stream", 8: "bwd_planes",
               9: "bwd_direct"}


def roi_variant(op: str, K: int, B: int, C: int, H: int, W: int, output_size=(7, 7), sampling_ratio: int = 2,
                want_argmax: bool = True, device=None) -> dict:
    """Kernel the RoI entry point ``op`` (a key of ROI_OPS) picks for this problem (host query, launches nothing).
    Without a CUDA device the choice is made for 148 SMs."""
    import ctypes
    out = (ctypes.c_int32 * 4)()
    args = (ROI_OPS[op], int(K), int(B), int(C), int(H), int(W), int(output_size[0]), int(output_size[1]),
            int(sampling_ratio), int(bool(want_argmax)), out)
    lib = _lib.load()
    if torch.cuda.is_available():
        with torch.cuda.device(device if device is not None else torch.cuda.current_device()):
            _lib.check(lib.frr_roi_variant(*args), "frr_roi_variant")
    else:
        _lib.check(lib.frr_roi_variant(*args), "frr_roi_variant")
    return dict(kernel=ROI_KERNELS[out[0]], cb=out[1], nz=out[2], smem=out[3])


# ------------------------------------------------------------------------------------------------
# RoIPool / RoIAlign (R1-R4): raw kernels + autograd functions
# ------------------------------------------------------------------------------------------------
def _feat_layout(feat: torch.Tensor):
    """Returns (tensor usable in place, channels_last flag).  NCHW-contiguous and channels_last memory are both
    consumed without a copy; anything else is made NCHW-contiguous."""
    if feat.dim() != 4:
        raise ValueError("features must be [B,C,H,W]")
    if feat.is_contiguous():
        return feat, 0
    if feat.is_contiguous(memory_format=torch.channels_last):
        return feat, 1
    return feat.contiguous(), 0


def convert_rois(rois, device=None) -> torch.Tensor:
    """torchvision's convention (TV ops/_utils.py:18-25): Tensor[K,5] or list of Tensor[L,4] (one per image)."""
    if isinstance(rois, (list, tuple)):
        parts = []
        for i, r in enumerate(rois):
            idx = torch.full((r.shape[0], 1), float(i), dtype=r.dtype, device=r.device)
            parts.append(torch.cat([idx, r], dim=1))
        rois = torch.cat(parts, dim=0) if parts else torch.zeros((0, 5), dtype=torch.float32, device=device)
    if rois.dim() != 2 or rois.shape[1] != 5:
        raise ValueError("rois must be Tensor[K,5] or a list of Tensor[L,4]")
    return rois


def rois5(rois, count, feat_hw, out=None):
    """models/model.py:104-110 for a batch: normalised rois [B,R,4] (+ int32 count [B] or None) -> [B*R,5] feature-map
    rois with the batch index; rows past count[b] are masked (index -1).  One kernel, no host synchronisation."""
    lib = _lib.load()
    rois = _req(rois, "rois")
    if rois.dim() != 3 or rois.shape[-1] != 4:
        raise ValueError("rois must be [B,R,4]")
    B, R = rois.shape[0], rois.shape[1]
    if count is not None:
        count = _req(count, "count", torch.int32)
    with torch.cuda.device(rois.device):
        if out is None:
            out = torch.empty((B * R, 5), dtype=torch.float32, device=rois.device)
        _lib.check(lib.frr_rois5(rois.data_ptr(), _ptr(count), B, R, float(feat_hw[1]), float(feat_hw[0]), out.data_ptr(),
                                 _stream()), "frr_rois5")
    return out


def roi_pool_forward(feat, rois5, output_size=(7, 7), spatial_scale: float = 1.0, want_argmax: bool = True):
    lib = _lib.load()
    feat = _req(feat, "features") if feat.is_contiguous() else feat
    if not feat.is_cuda or feat.dtype != torch.float32:
        raise ValueError("features must be a CUDA fp32 tensor: the region stage has no CPU path")
    feat, cl = _feat_layout(feat)
    rois5 = _req(rois5, "rois")
    B, C, H, W = feat.shape
    K = rois5.shape[0]
    PH, PW = int(output_size[0]), int(output_size[1])
    with torch.cuda.device(feat.device):
        out = torch.empty((K, C, PH, PW), dtype=torch.float32, device=feat.device)
        arg = torch.empty((K, C, PH, PW), dtype=torch.int32, device=feat.device) if want_argmax else None
        _lib.check(lib.frr_roi_pool_fwd(feat.data_ptr(), rois5.data_ptr(), K, B, C, H, W, PH, PW, float(spatial_scale), cl,
                                        out.data_ptr(), _ptr(arg), _stream()), "frr_roi_pool_fwd")
    return out, arg


def roi_pool_backward(grad_out, argmax, rois5, feat_shape, spatial_scale: float = 1.0, channels_last: bool = False):
    lib = _lib.load()
    grad_out = _req(grad_out, "grad_out")
    argmax = _req(argmax, "argmax", torch.int32)
    rois5 = _req(rois5, "rois")
    B, C, H, W = feat_shape
    K, _, PH, PW = grad_out.shape
    with torch.cuda.device(grad_out.device):
        gin = torch.empty((B, C, H, W), dtype=torch.float32, device=grad_out.device,
                          memory_format=torch.channels_last if channels_last else torch.contiguous_format)
        _lib.check(lib.frr_roi_pool_bwd(grad_out.data_ptr(), argmax.data_ptr(), rois5.data_ptr(), K, B, C, H, W, PH, PW,
                                        float(spatial_scale), int(channels_last), gin.data_ptr(), _stream()),
                   "frr_roi_pool_bwd")
    return gin


def roi_align_forward(feat, rois5, output_size=(7, 7), spatial_scale: float = 1.0, sampling_ratio: int = 2,
                      aligned: bool = False, out=None):
    """``out``: write into an existing [K,C,PH,PW] tensor (rows of rois with a negative batch index are left untouched)."""
    lib = _lib.load()
    if not feat.is_cuda or feat.dtype != torch.float32:
        raise ValueError("features must be a CUDA fp32 tensor: the region stage has no CPU path")
    feat, cl = _feat_layout(feat)
    rois5 = _req(rois5, "rois")
    B, C, H, W = feat.shape
    K = rois5.shape[0]
    PH, PW = int(output_size[0]), int(output_size[1])
    with torch.cuda.device(feat.device):
        if out is None:
            out = torch.empty((K, C, PH, PW), dtype=torch.float32, device=feat.device)
        elif tuple(out.shape) != (K, C, PH, PW) or not out.is_contiguous() or out.dtype != torch.float32:
            raise ValueError("roi_align_forward: out must be a contiguous fp32 [K,C,PH,PW] tensor")
        _lib.check(lib.frr_roi_align_fwd(feat.data_ptr(), rois5.data_ptr(), K, B, C, H, W, PH, PW, float(spatial_scale),
                                         int(sampling_ratio), int(aligned), cl, out.data_ptr(), _stream()),
                   "frr_roi_align_fwd")
    return out


def roi_align_backward(grad_out, rois5, feat_shape, spatial_scale: float = 1.0, sampling_ratio: int = 2,
                       aligned: bool = False, channels_last: bool = False):
    lib = _lib.load()
    grad_out = _req(grad_out, "grad_out")
    rois5 = _req(rois5, "rois")
    B, C, H, W = feat_shape
    K, _, PH, PW = grad_out.shape
    with torch.cuda.device(grad_out.device):
        gin = torch.empty((B, C, H, W), dtype=torch.float32, device=grad_out.device,
                          memory_format=torch.channels_last if channels_last else torch.contiguous_format)
        _lib.check(lib.frr_roi_align_bwd(grad_out.data_ptr(), rois5.data_ptr(), K, B, C, H, W, PH, PW, float(spatial_scale),
                                         int(sampling_ratio), int(aligned), int(channels_last), gin.data_ptr(), _stream()),
                   "frr_roi_align_bwd")
    return gin


class _RoIPoolFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, rois5, output_size, spatial_scale):
        feat_l, cl = _feat_layout(feat)
        out, arg = roi_pool_forward(feat_l, rois5, output_size, spatial_scale, want_argmax=True)
        ctx.save_for_backward(rois5, arg)
        ctx.meta = (tuple(feat.shape), float(spatial_scale), bool(cl))
        return out

    @staticmethod
    def backward(ctx, grad_out):
        rois5, arg = ctx.saved_tensors
        shape, scale, cl = ctx.meta
        return roi_pool_backward(grad_out.contiguous(), arg, rois5, shape, scale, cl), None, None, None


class _RoIAlignFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, rois5, output_size, spatial_scale, sampling_ratio, aligned):
        feat_l, cl = _feat_layout(feat)
        out = roi_align_forward(feat_l, rois5, output_size, spatial_scale, sampling_ratio, aligned)
        ctx.save_for_backward(rois5)
        ctx.meta = (tuple(feat.shape), float(spatial_scale), int(sampling_ratio), bool(aligned), bool(cl))
        return out

    @staticmethod
    def backward(ctx, grad_out):
        (rois5,) = ctx.saved_tensors
        shape, scale, sr, al, cl = ctx.meta
        return roi_align_backward(grad_out.contiguous(), rois5, shape, scale, sr, al, cl), None, None, None, None, None


def roi_pool(input, boxes, output_size, spatial_scale: float = 1.0):
    """Drop-in for torchvision.ops.roi_pool (differentiable w.r.t. ``input``)."""
    if isinstance(output_size, int):
        output_size = (output_size, output_size)
    rois5 = convert_rois(boxes, input.device).to(torch.float32)
    return _RoIPoolFn.apply(input, rois5.contiguous(), tuple(output_size), float(spatial_scale))


def roi_align(input, boxes, output_size, spatial_scale: float = 1.0, sampling_ratio: int = -1, aligned: bool = False):
    """Drop-in for torchvision.ops.roi_align (differentiable w.r.t. ``input``)."""
    if isinstance(output_size, int):
        output_size = (output_size, output_size)
    rois5 = convert_rois(boxes, input.device).to(torch.float32)
    return _RoIAlignFn.apply(input, rois5.contiguous(), tuple(output_size), float(spatial_scale), int(sampling_ratio),
                             bool(aligned))


# ------------------------------------------------------------------------------------------------
# target makers (T1-T4): raw two-phase kernels; the host sampling logic lives in targets.py
# ------------------------------------------------------------------------------------------------
_STD4 = np.array([0.1, 0.1, 0.2, 0.2], dtype=np.float32)       # models/model.py:176,372


VARIANTS = {   # (iou_eps, inside_only, tie_inclusive): models/model.py vs models/new_model.py target makers
    "vgg": (float(np.float32(1e-5)), 1, 0),
    "fpn": (0.0, 0, 1),
}


def rpn_targets_assign(gt, gt_count, N, image_hw=None, anchors=None, stride=16, table=None, neg_thr=0.3, pos_thr=0.7,
                       variant: str = "vgg"):
    lib = _lib.load()
    eps, inside_only, tie_inclusive = VARIANTS[variant]
    gt = _req(gt, "gt")
    if gt.dim() != 3 or gt.shape[-1] != 4:
        raise ValueError("gt must be [B,Gmax,4]")
    B, G = gt.shape[0], gt.shape[1]
    if G == 0:
        raise IndexError("max(): Expected reduction dim 1 to have non-zero size")   # models/model.py:199
    if gt_count is not None:
        gt_count = _req(gt_count, "gt_count", torch.int32)
    keep, tptr, A = _table_arg(table)
    if anchors is not None:
        anchors = _req(anchors, "anchors")
        H = W = 0
    else:
        H, W = int(image_hw[0]), int(image_hw[1])
    dev = gt.device
    with torch.cuda.device(dev):
        ws = dict(iou_max=torch.empty((B, N), dtype=torch.float32, device=dev),
                  argmax=torch.empty((B, N), dtype=torch.int32, device=dev),
                  label8=torch.empty((B, N), dtype=torch.int8, device=dev),
                  pos_list=torch.empty((B, N), dtype=torch.int32, device=dev),
                  neg_list=torch.empty((B, N), dtype=torch.int32, device=dev),
                  counts=torch.empty((B, 2), dtype=torch.int32, device=dev))
        _lib.check(lib.frr_rpn_targets_assign(gt.data_ptr(), _ptr(gt_count), B, G, _ptr(anchors), tptr, A, H, W, stride, N,
                                              float(np.float32(neg_thr)), float(np.float32(pos_thr)), eps, inside_only,
                                              tie_inclusive, ws["iou_max"].data_ptr(), ws["argmax"].data_ptr(), ws["label8"].data_ptr(),
                                              ws["pos_list"].data_ptr(), ws["neg_list"].data_ptr(), ws["counts"].data_ptr(),
                                              _stream()), "frr_rpn_targets_assign")
    ws.update(gt=gt, anchors=anchors, geom=(H, W, stride, table, N))
    return ws


def rpn_targets_finalize(ws, disable=None, disable_off=None):
    lib = _lib.load()
    gt, anchors = ws["gt"], ws["anchors"]
    H, W, stride, table, N = ws["geom"]
    keep, tptr, A = _table_arg(table)
    B, G = gt.shape[0], gt.shape[1]
    dev = gt.device
    with torch.cuda.device(dev):
        labels = torch.empty((B, N), dtype=torch.int64, device=dev)
        reg = torch.empty((B, N, 4), dtype=torch.float32, device=dev)
        _lib.check(lib.frr_rpn_targets_finalize(gt.data_ptr(), B, G, _ptr(anchors), tptr, A, H, W, stride, N,
                                                ws["argmax"].data_ptr(), ws["label8"].data_ptr(), ws["pos_list"].data_ptr(),
                                                ws["neg_list"].data_ptr(), _ptr(disable), _ptr(disable_off),
                                                labels.data_ptr(), reg.data_ptr(), _stream()), "frr_rpn_targets_finalize")
    return labels, reg


def frcnn_targets_assign(rois, roi_count, gt, gt_count, fg_thr=0.5, variant: str = "vgg"):
    lib = _lib.load()
    eps = VARIANTS[variant][0]
    rois = _req(rois, "rois")
    gt = _req(gt, "gt")
    B, R = rois.shape[0], rois.shape[1]
    G = gt.shape[1]
    if G == 0:
        raise IndexError("max(): Expected reduction dim 1 to have non-zero size")
    if roi_count is not None:
        roi_count = _req(roi_count, "roi_count", torch.int32)
    if gt_count is not None:
        gt_count = _req(gt_count, "gt_count", torch.int32)
    M = R + G
    dev = rois.device
    with torch.cuda.device(dev):
        ws = dict(iou_max=torch.empty((B, M), dtype=torch.float32, device=dev),
                  argmax=torch.empty((B, M), dtype=torch.int32, device=dev),
                  label8=torch.empty((B, M), dtype=torch.int8, device=dev),
                  pos_list=torch.empty((B, M), dtype=torch.int32, device=dev),
                  neg_list=torch.empty((B, M), dtype=torch.int32, device=dev),
                  counts=torch.empty((B, 2), dtype=torch.int32, device=dev))
        _lib.check(lib.frr_frcnn_targets_assign(rois.data_ptr(), _ptr(roi_count), B, R, gt.data_ptr(), _ptr(gt_count), G,
                                                float(np.float32(fg_thr)), eps, ws["iou_max"].data_ptr(), ws["argmax"].data_ptr(),
                                                ws["label8"].data_ptr(), ws["pos_list"].data_ptr(), ws["neg_list"].data_ptr(),
                                                ws["counts"].data_ptr(), _stream()), "frr_frcnn_targets_assign")
    ws.update(rois=rois, roi_count=roi_count, gt=gt)
    return ws


def frcnn_targets_finalize(ws, gt_label, sel, sel_n, std=_STD4, label_offset: int = 1):
    lib = _lib.load()
    rois, gt = ws["rois"], ws["gt"]
    gt_label = _req(gt_label, "gt_label", torch.int64)
    sel = _req(sel, "sel", torch.int32)
    sel_n = _req(sel_n, "sel_n", torch.int32)
    B, R, G, S = rois.shape[0], rois.shape[1], gt.shape[1], sel.shape[1]
    std = np.ascontiguousarray(std, dtype=np.float32)
    dev = rois.device
    with torch.cuda.device(dev):
        cls = torch.empty((B, S), dtype=torch.int64, device=dev)
        reg = torch.empty((B, S, 4), dtype=torch.float32, device=dev)
        srois = torch.empty((B, S, 4), dtype=torch.float32, device=dev)
        kidx = torch.empty((B, S), dtype=torch.int32, device=dev)
        _lib.check(lib.frr_frcnn_targets_finalize(rois.data_ptr(), _ptr(ws["roi_count"]), B, R, gt.data_ptr(),
                                                  gt_label.data_ptr(), G, ws["argmax"].data_ptr(), ws["pos_list"].data_ptr(),
                                                  ws["neg_list"].data_ptr(), sel.data_ptr(), sel_n.data_ptr(), S,
                                                  std.ctypes.data, int(label_offset), cls.data_ptr(), reg.data_ptr(), srois.data_ptr(),
                                                  kidx.data_ptr(), _stream()), "frr_frcnn_targets_finalize")
    return cls, reg, srois, kidx


def sample_targets(mt_state, ws_rpn=None, ws_frcnn=None, rpn_batch: int = 256, rpn_max_pos: int = 128,
                   frcnn_batch: int = 128, frcnn_max_pos: int = 32):
    """The reference's torch.randperm sampling replayed on the device (``frr_sample_targets``): ``mt_state`` is the
    uint32 [626] device copy of torch's CPU mt19937 state (``targets.DeviceGenerator``), advanced in place.  Edits
    ``ws_rpn['label8']`` in place and returns (sel int32 [B,frcnn_batch], sel_n int32 [B,2]) for the Fast R-CNN finalize
    (None, None when ``ws_frcnn`` is None).  No host synchronisation."""
    lib = _lib.load()
    if ws_rpn is None and ws_frcnn is None:
        raise ValueError("sample_targets: nothing to sample")
    ref = ws_rpn if ws_rpn is not None else ws_frcnn
    dev = ref["counts"].device
    B = ref["counts"].shape[0]
    if mt_state.device != dev or mt_state.dtype != torch.int32 or mt_state.numel() != 626:
        raise ValueError("mt_state must be an int32 [626] tensor on the device of the targets")
    S = max(rpn_batch if ws_rpn is not None else 0, frcnn_batch if ws_frcnn is not None else 0)
    with torch.cuda.device(dev):
        jobs = torch.empty((B, 4, 4), dtype=torch.int32, device=dev)
        draws = torch.empty((B, 4, S), dtype=torch.int32, device=dev)
        sel = sel_n = None
        if ws_frcnn is not None:
            sel = torch.zeros((B, frcnn_batch), dtype=torch.int32, device=dev)
            sel_n = torch.zeros((B, 2), dtype=torch.int32, device=dev)
        N = ws_rpn["label8"].shape[1] if ws_rpn is not None else 0
        _lib.check(lib.frr_sample_targets(_ptr(ws_rpn["counts"]) if ws_rpn is not None else None,
                                          _ptr(ws_frcnn["counts"]) if ws_frcnn is not None else None, B, int(rpn_batch),
                                          int(rpn_max_pos), int(frcnn_batch), int(frcnn_max_pos), mt_state.data_ptr(), N,
                                          _ptr(ws_rpn["label8"]) if ws_rpn is not None else None,
                                          _ptr(ws_rpn["pos_list"]) if ws_rpn is not None else None,
                                          _ptr(ws_rpn["neg_list"]) if ws_rpn is not None else None, _ptr(sel), _ptr(sel_n),
                                          int(frcnn_batch), jobs.data_ptr(), draws.data_ptr(), S, _stream()),
                   "frr_sample_targets")
    return sel, sel_n


# ------------------------------------------------------------------------------------------------
# loss side (losses/loss.py:5-59 + the class-row gather of models/model.py:340-341)
# ------------------------------------------------------------------------------------------------
RPN_BETA, FRCNN_BETA = float(np.float32(1 / 9)), 1.0      # losses/loss.py:21,47


class _RegionLossFn(torch.autograd.Function):
    """One kernel computes the four losses and, for a unit upstream gradient, their gradients w.r.t. the predictions;
    backward only scales the saved gradients by the upstream values."""

    @staticmethod
    def forward(ctx, rpn_cls, rpn_reg, frc_cls, frc_reg, rpn_tcls, rpn_treg, frc_tcls, frc_treg):
        lib = _lib.load()
        have_rpn, have_frc = rpn_cls is not None, frc_cls is not None
        ref = rpn_cls if have_rpn else frc_cls
        dev = ref.device
        B = ref.shape[0]
        N = rpn_cls.shape[1] if have_rpn else 0
        S, C = (frc_cls.shape[1], frc_cls.shape[2]) if have_frc else (0, 0)
        CR = frc_reg.shape[2] if have_frc else 0
        need = [have_rpn and ctx.needs_input_grad[0], have_rpn and ctx.needs_input_grad[1],
                have_frc and ctx.needs_input_grad[2], have_frc and ctx.needs_input_grad[3]]
        with torch.cuda.device(dev):
            loss = torch.empty((B, 5), dtype=torch.float32, device=dev)
            grads = [torch.empty_like(t) if n else None for t, n in zip((rpn_cls, rpn_reg, frc_cls, frc_reg), need)]
            _lib.check(lib.frr_region_loss(_ptr(rpn_cls), _ptr(rpn_reg), _ptr(rpn_tcls), _ptr(rpn_treg), B, N, _ptr(frc_cls),
                                           _ptr(frc_reg), _ptr(frc_tcls), _ptr(frc_treg), S, C, CR, RPN_BETA, FRCNN_BETA,
                                           loss.data_ptr(), _ptr(grads[0]), _ptr(grads[1]), _ptr(grads[2]), _ptr(grads[3]),
                                           _stream()), "frr_region_loss")
        ctx.grads = grads
        return loss

    @staticmethod
    def backward(ctx, g):            # g [B,5]: upstream of (total, rpn_cls, rpn_reg, frcnn_cls, frcnn_reg)
        out = []
        for j, saved in enumerate(ctx.grads):
            if saved is None:
                out.append(None)
                continue
            up = (g[:, 0] + g[:, 1 + j]).reshape((-1,) + (1,) * (saved.dim() - 1))
            out.append(saved * up)
        return tuple(out) + (None, None, None, None)


def region_loss(rpn_cls=None, rpn_reg=None, rpn_target_cls=None, rpn_target_reg=None, frcnn_cls=None, frcnn_reg=None,
                frcnn_target_cls=None, frcnn_target_reg=None):
    """Batched FRCNNLoss (losses/loss.py:62-82): per image (total, rpn_cls, rpn_reg, frcnn_cls, frcnn_reg) -> [B,5],
    differentiable w.r.t. the four prediction tensors.  rpn_cls [B,N,2], rpn_reg [B,N,4], rpn_target_cls int64 [B,N],
    rpn_target_reg [B,N,4]; frcnn_cls [B,S,C], frcnn_reg [B,S,C,4] (or [B,S,C*4]: the head output, the class row is
    gathered in the kernel, models/model.py:340-341) or [B,S,4] (already gathered), frcnn_target_cls int64 [B,S]
    (negative = padding), frcnn_target_reg [B,S,4].  Either half may be omitted."""
    if rpn_cls is None and frcnn_cls is None:
        raise ValueError("region_loss: nothing to compute")
    if rpn_cls is not None:
        rpn_cls, rpn_reg, rpn_target_reg = _req(rpn_cls, "rpn_cls"), _req(rpn_reg, "rpn_reg"), _req(rpn_target_reg, "rpn_target_reg")
        rpn_target_cls = _req(rpn_target_cls, "rpn_target_cls", torch.int64)
        B, N = rpn_cls.shape[0], rpn_cls.shape[1]
        if tuple(rpn_cls.shape) != (B, N, 2) or tuple(rpn_reg.shape) != (B, N, 4) or tuple(rpn_target_cls.shape) != (B, N) \
                or tuple(rpn_target_reg.shape) != (B, N, 4):
            raise ValueError("region_loss: RPN tensors must be [B,N,2], [B,N,4], [B,N], [B,N,4]")
    if frcnn_cls is not None:
        frcnn_cls, frcnn_reg = _req(frcnn_cls, "frcnn_cls"), _req(frcnn_reg, "frcnn_reg")
        frcnn_target_cls = _req(frcnn_target_cls, "frcnn_target_cls", torch.int64)
        frcnn_target_reg = _req(frcnn_target_reg, "frcnn_target_reg")
        B, S, C = frcnn_cls.shape
        if frcnn_reg.numel() == B * S * C * 4:
            frcnn_reg = frcnn_reg.reshape(B, S, C, 4)
        elif frcnn_reg.numel() == B * S * 4:
            frcnn_reg = frcnn_reg.reshape(B, S, 1, 4)
        else:
            raise ValueError("region_loss: frcnn_reg must hold C or 1 rows of 4 per sample")
        if tuple(frcnn_target_cls.shape) != (B, S) or tuple(frcnn_target_reg.shape) != (B, S, 4):
            raise ValueError("region_loss: Fast R-CNN targets must be [B,S] and [B,S,4]")
    return _RegionLossFn.apply(rpn_cls, rpn_reg, frcnn_cls, frcnn_reg, rpn_target_cls, rpn_target_reg, frcnn_target_cls,
                               frcnn_target_reg)


# ------------------------------------------------------------------------------------------------
# detection post-processing (D1, D2)
# ------------------------------------------------------------------------------------------------
def decode_classwise(cls_logits, reg, rois, num_classes: int, std=_STD4):
    """cls [rows,C], reg [rows,4C], rois [rows,4] -> prob [rows,C], boxes [rows,4C] (clamped to [0,1])."""
    lib = _lib.load()
    cls_logits = _req(cls_logits, "cls_logits")
    reg = _req(reg, "reg")
    rois = _req(rois, "rois")
    rows, C = cls_logits.shape[0], int(num_classes)
    if cls_logits.shape[1] != C or reg.numel() != rows * C * 4 or rois.numel() != rows * 4:
        raise ValueError("decode_classwise: shape mismatch")
    std = np.ascontiguousarray(std, dtype=np.float32)
    dev = cls_logits.device
    with torch.cuda.device(dev):
        prob = torch.empty((rows, C), dtype=torch.float32, device=dev)
        boxes = torch.empty((rows, C * 4), dtype=torch.float32, device=dev)
        _lib.check(lib.frr_decode_classwise(cls_logits.data_ptr(), reg.data_ptr(), rois.data_ptr(), rows, C, std.ctypes.data,
                                            prob.data_ptr(), boxes.data_ptr(), _stream()), "frr_decode_classwise")
    return prob, boxes


def class_nms(prob, boxes, num_classes: int, score_thres: float = 0.05, iou_thr: float = 0.3, roi_count=None, cap=None):
    """prob [B,R,C], boxes [B,R,4C] -> det_boxes [B,cap,4], det_labels int32 [B,cap], det_scores [B,cap], count [B]."""
    lib = _lib.load()
    prob = _req(prob, "prob")
    boxes = _req(boxes, "boxes")
    B, R, C = prob.shape[0], prob.shape[1], int(num_classes)
    if prob.shape[2] != C or boxes.numel() != B * R * C * 4:
        raise ValueError("class_nms: shape mismatch")
    if roi_count is not None:
        roi_count = _req(roi_count, "roi_count", torch.int32)
    cap = R * (C - 1) if cap is None else int(cap)
    dev = prob.device
    with torch.cuda.device(dev):
        nbytes = int(lib.frr_class_nms_workspace_bytes(B, R, C))
        ws = torch.empty((nbytes + 256,), dtype=torch.uint8, device=dev)
        off = (-ws.data_ptr()) % 256
        db = torch.empty((B, cap, 4), dtype=torch.float32, device=dev)
        dl = torch.empty((B, cap), dtype=torch.int32, device=dev)
        ds = torch.empty((B, cap), dtype=torch.float32, device=dev)
        dc = torch.empty((B,), dtype=torch.int32, device=dev)
        _lib.check(lib.frr_class_nms(prob.data_ptr(), boxes.data_ptr(), _ptr(roi_count), B, R, C,
                                     float(np.float32(score_thres)), float(iou_thr), cap, db.data_ptr(), dl.data_ptr(),
                                     ds.data_ptr(), dc.data_ptr(), ws.data_ptr() + off, nbytes, _stream()), "frr_class_nms")
    return db, dl, ds, dc


def pack_detections(det_boxes, det_labels, det_scores, det_count, max_det: int, image_wh=None, xywh: bool = False):
    """Evaluation hand-off (test.py:68-88, evaluation/coco_eval.py:156-158): [B,cap,4] / [B,cap] / [B,cap] / [B] ->
    ([B,max_det,6] rows (x, y, x2|w, y2|h, score, label) scaled by ``image_wh [B,2]`` = (w, h), int32 counts [B])."""
    lib = _lib.load()
    det_boxes = _req(det_boxes, "det_boxes")
    det_labels = _req(det_labels, "det_labels", torch.int32)
    det_scores = _req(det_scores, "det_scores")
    det_count = _req(det_count, "det_count", torch.int32)
    if image_wh is not None:
        image_wh = _req(image_wh, "image_wh")
    B, cap = det_labels.shape
    dev = det_boxes.device
    with torch.cuda.device(dev):
        out = torch.empty((B, int(max_det), 6), dtype=torch.float32, device=dev)
        cnt = torch.empty((B,), dtype=torch.int32, device=dev)
        _lib.check(lib.frr_pack_detections(det_boxes.data_ptr(), det_labels.data_ptr(), det_scores.data_ptr(),
                                           det_count.data_ptr(), B, cap, int(max_det), _ptr(image_wh), int(bool(xywh)),
                                           out.data_ptr(), cnt.data_ptr(), _stream()), "frr_pack_detections")
    return out, cnt


# ------------------------------------------------------------------------------------------------
# MultiScaleRoIAlign (models/new_model.py:127,143; TV ops/poolers.py)
# ------------------------------------------------------------------------------------------------
def infer_scales(features, image_shapes):
    """TV ops/poolers.py ``_setup_scales`` / ``_infer_scale``: scale_l = 2 ** round(log2(feat_dim0 / image_dim0)) with
    image_dim0 = max over ``image_shapes`` of their first entry (used exactly as the caller passes them; the reference
    passes (w, h)).  Returns (scales, k_min, k_max)."""
    import math
    if not image_shapes:
        raise ValueError("images list should not be empty")
    d0 = max(int(s[0]) for s in image_shapes)
    scales = [2.0 ** float(round(math.log2(float(f.shape[-2]) / float(d0)))) for f in features]
    return scales, int(-math.log2(scales[0])), int(-math.log2(scales[-1]))


def fpn_level_rois(rois5, k_min: int, k_max: int, canonical_scale: float = 224.0, canonical_level: int = 4):
    """LevelMapper on the device: (levels int32 [K], rois_per_level [L,K,5] with foreign rois masked by batch index -1)."""
    lib = _lib.load()
    rois5 = _req(rois5, "rois")
    K, L = rois5.shape[0], k_max - k_min + 1
    with torch.cuda.device(rois5.device):
        levels = torch.empty((K,), dtype=torch.int32, device=rois5.device)
        per = torch.empty((L, K, 5), dtype=torch.float32, device=rois5.device)
        _lib.check(lib.frr_fpn_level_rois(rois5.data_ptr(), K, int(k_min), int(k_max), int(canonical_level),
                                          float(canonical_scale), L, levels.data_ptr(), per.data_ptr(), _stream()),
                   "frr_fpn_level_rois")
    return levels, per


class _MultiScaleRoIAlignFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rois5, output_size, sampling_ratio, scales, k_min, k_max, canonical_scale, canonical_level, *feats):
        K, C = rois5.shape[0], feats[0].shape[1]
        levels, per = fpn_level_rois(rois5, k_min, k_max, canonical_scale, canonical_level)
        out = torch.empty((K, C, output_size[0], output_size[1]), dtype=torch.float32, device=rois5.device)
        lay = []
        for l, f in enumerate(feats):
            f_l, cl = _feat_layout(f)
            lay.append(bool(cl))
            roi_align_forward(f_l, per[l], output_size, scales[l], sampling_ratio, False, out=out)
        ctx.save_for_backward(per)
        ctx.meta = ([tuple(f.shape) for f in feats], list(scales), int(sampling_ratio), lay)
        ctx.mark_non_differentiable(levels)
        return out, levels

    @staticmethod
    def backward(ctx, grad_out, _grad_levels):
        (per,) = ctx.saved_tensors
        shapes, scales, sr, lay = ctx.meta
        go = grad_out.contiguous()
        grads = [roi_align_backward(go, per[l], shapes[l], scales[l], sr, False, lay[l]) for l in range(len(shapes))]
        return (None,) * 8 + tuple(grads)


def multiscale_roi_align(features, boxes, image_shapes, output_size=7, sampling_ratio: int = 2,
                         canonical_scale: float = 224.0, canonical_level: int = 4, return_levels: bool = False):
    """Drop-in for ``torchvision.ops.MultiScaleRoIAlign(featmap_names, output_size, sampling_ratio)(x, boxes,
    image_shapes)`` as called at models/new_model.py:127,143: ``features`` = list (or dict values, in order) of
    [B,C,Hl,Wl] maps, ``boxes`` = Tensor[K,5] or list of Tensor[L,4] in image coordinates.  One level-assignment
    kernel + one RoIAlign launch per level, all writing one [K,C,7,7] output; differentiable w.r.t. the features."""
    if isinstance(features, dict):
        features = list(features.values())
    features = list(features)
    if isinstance(output_size, int):
        output_size = (output_size, output_size)
    rois5 = convert_rois(boxes, features[0].device).to(torch.float32).contiguous()
    scales, k_min, k_max = infer_scales(features, image_shapes)
    if len(features) == 1:
        out = roi_align(features[0], rois5, output_size, scales[0], sampling_ratio, False)
        return (out, torch.zeros((rois5.shape[0],), dtype=torch.int32, device=rois5.device)) if return_levels else out
    out, levels = _MultiScaleRoIAlignFn.apply(rois5, tuple(output_size), int(sampling_ratio), tuple(scales), k_min, k_max,
                                              float(canonical_scale), int(canonical_level), *features)
    return (out, levels) if return_levels else out
