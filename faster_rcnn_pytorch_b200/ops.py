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


def _check(t: torch.Tensor, name: str, dtype=torch.float32, shape=None, device=None, contiguous: bool = False):
    """The contract of a tensor handed to libfrr as a bare pointer: a CUDA tensor of ``dtype``, on ``device`` (the launch
    device) and of ``shape`` (a tuple of ints, None = any size in that dimension) when given, and already contiguous when
    ``contiguous`` is set (where a copy would be wrong: a tensor written in place, whose copy would not reach the caller,
    or the input of a plan that allocates nothing).  Returns ``t``; raises TypeError for a non-tensor, ValueError for any
    other mismatch."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if device is None or t.device != device:              # on the CUDA ``device``: CUDA needs no test of its own
        if not t.is_cuda:
            raise ValueError(f"{name} must be a CUDA tensor: the region stage has no CPU path")
        if device is not None:
            raise ValueError(f"{name} must be on {device}, the device of the launch, got {t.device}")
    if t.dtype != dtype:
        raise ValueError(f"{name} must be {dtype}, got {t.dtype}")
    if shape is not None:
        s = t.shape                                       # a full tuple matches in one comparison
        if s != shape and (len(s) != len(shape) or [d for d, w in zip(s, shape) if w is not None and d != w]):
            want = ",".join("*" if w is None else str(w) for w in shape)
            raise ValueError(f"{name} must be [{want}], got {list(s)}")
    if contiguous and not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return t


def _req(t: torch.Tensor, name: str, dtype=torch.float32, shape=None, device=None):
    """An input a kernel reads: ``t`` checked by ``_check`` and made contiguous."""
    return _check(t, name, dtype, shape, device).contiguous()


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


def is_sized(image_hw) -> bool:
    """True when ``image_hw`` gives one (H, W) per image ([B,2]: a mixed-size batch) rather than one for the batch."""
    if isinstance(image_hw, torch.Tensor):
        return image_hw.dim() == 2
    return image_hw is not None and np.ndim(image_hw) == 2


def sized_hw(image_hw, B: int, grid_hw, stride: int, device) -> torch.Tensor:
    """Per-image sizes of a mixed-size batch as the int32 [B,2] (H, W) device tensor the *_sized kernels read.

    A CUDA tensor is used as it is (int32, [B,2]): its values are read by the kernels when they run, so one captured CUDA
    graph serves every mix of sizes written into it, and the kernels clamp each image's grid (H // stride, W // stride) to
    ``grid_hw``.  Host sizes (CPU tensor, numpy array, list of pairs) are checked here, where that costs nothing: every
    image's grid must fit ``grid_hw``, else ValueError, and they are copied to ``device``."""
    gh, gw = int(grid_hw[0]), int(grid_hw[1])
    if isinstance(image_hw, torch.Tensor) and image_hw.is_cuda:
        dev = torch.device(device)
        if dev.index is None:                  # "cuda": the current device, where torch allocates for it
            dev = torch.device(dev.type, torch.cuda.current_device())
        return _req(image_hw, "image_hw", torch.int32, (B, 2), dev)
    hw = np.asarray(image_hw.numpy() if isinstance(image_hw, torch.Tensor) else image_hw, dtype=np.int64)
    if hw.shape != (B, 2):
        raise ValueError(f"image_hw must be [{B},2] (H, W) per image, got shape {hw.shape}")
    if (hw < 0).any() or (hw[:, 0] // stride > gh).any() or (hw[:, 1] // stride > gw).any():
        raise ValueError(f"image_hw: every image's grid (H // {stride}, W // {stride}) must fit the padded grid {gh}x{gw}")
    return torch.from_numpy(hw.astype(np.int32)).to(device)


def rpn_decode(reg, cls, image_hw=None, anchors=None, stride: int = 16, table=None, min_size: float = _MIN_SIZE,
               grid_hw=None):
    """Fused A2+P1+P2+P3.  reg [B,N,4]; cls [B,N,2] logits or [B,N] scores.
    Returns boxes [B,N,4], scores [B,N], valid uint8 [B,N].

    Mixed-size batch: ``image_hw`` [B,2] (one (H, W) per image, see ``sized_hw``) and ``grid_hw`` = the padded grid in
    cells, N = grid_h * grid_w * A.  Each image is decoded exactly as alone at its own size; its padding cells get
    box 0, score 0, valid 0."""
    lib = _lib.load()
    reg = _req(reg, "reg", shape=(None, None, 4))
    B, N, dev = reg.shape[0], reg.shape[1], reg.device
    logits = isinstance(cls, torch.Tensor) and cls.dim() == 3
    cls = _req(cls, "cls", shape=(B, N, 2) if logits else (B, N), device=dev)
    keep, tptr, A = _table_arg(table)
    if is_sized(image_hw):
        if anchors is not None or grid_hw is None:
            raise ValueError("rpn_decode: per-image sizes need grid_hw and generated anchors")
        hw = sized_hw(image_hw, B, grid_hw, stride, dev)
        with torch.cuda.device(dev):
            boxes = torch.empty((B, N, 4), dtype=torch.float32, device=dev)
            scores = torch.empty((B, N), dtype=torch.float32, device=dev)
            valid = torch.empty((B, N), dtype=torch.uint8, device=dev)
            _lib.check(lib.frr_rpn_decode_sized(reg.data_ptr(), cls.data_ptr(), int(logits), tptr, A, hw.data_ptr(),
                                                int(grid_hw[0]), int(grid_hw[1]), stride, float(min_size), boxes.data_ptr(),
                                                scores.data_ptr(), valid.data_ptr(), B, N, _stream()), "frr_rpn_decode_sized")
        return boxes, scores, valid
    if anchors is not None:
        anchors = _req(anchors, "anchors", shape=(N, 4), device=dev)
        H = W = 0
    else:
        if image_hw is None:
            raise ValueError("image_hw is required when anchors are generated in-kernel")
        H, W = int(image_hw[0]), int(image_hw[1])
    with torch.cuda.device(dev):
        boxes = torch.empty((B, N, 4), dtype=torch.float32, device=dev)
        scores = torch.empty((B, N), dtype=torch.float32, device=dev)
        valid = torch.empty((B, N), dtype=torch.uint8, device=dev)
        _lib.check(lib.frr_rpn_decode(reg.data_ptr(), cls.data_ptr(), int(logits), _ptr(anchors), tptr, A, H, W, stride,
                                      float(min_size), boxes.data_ptr(), scores.data_ptr(), valid.data_ptr(), B, N,
                                      _stream()), "frr_rpn_decode")
    return boxes, scores, valid


def topk_desc(scores, k: int, valid=None, boxes=None, want_cidx: bool = False, ctas_per_image: int = 0):
    """P4.  scores [B,N] -> dict(scores [B,k], idx int32 [B,k], cidx, boxes [B,k,4], count int32 [B]).
    ``ctas_per_image``: 0 = automatic (a 2-CTA cluster per image for small batches), 1 = one CTA per image."""
    lib = _lib.load()
    scores = _req(scores, "scores", shape=(None, None))
    (B, N), dev = scores.shape, scores.device
    if valid is not None:
        valid = _req(valid, "valid", torch.uint8, (B, N), dev)
    if boxes is not None:
        boxes = _req(boxes, "boxes", shape=(B, N, 4), device=dev)
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
               cluster_size: int = 0, threads: int = 0, unit_boxes: bool = False, first_chunk: int = 0,
               max_chunk: int = 0, lanes_screen: int = 0, lanes_pairs: int = 0):
    """N1 on score-sorted boxes [B,n,4].  Returns keep int32 [B,max_keep] (-1 padded), count int32 [B],
    rois [B,max_keep,4] (zero padded) or None.  ``unit_boxes``: the caller guarantees coordinates in [0,1]
    (enables a cheaper, result-identical screening test).  ``first_chunk``, ``max_chunk``, ``lanes_screen``,
    ``lanes_pairs``: settings of the bucketed variant, 0 = automatic; results do not depend on them."""
    lib = _lib.load()
    boxes = _req(boxes, "boxes", shape=(None, None, 4))
    B, n, dev = boxes.shape[0], boxes.shape[1], boxes.device
    mk = n if max_keep is None else int(max_keep)
    if counts is not None:
        counts = _req(counts, "counts", torch.int32, (B,), dev)
    with torch.cuda.device(dev):
        keep = torch.empty((B, mk), dtype=torch.int32, device=dev)
        cnt = torch.empty((B,), dtype=torch.int32, device=dev)
        rois = torch.empty((B, mk, 4), dtype=torch.float32, device=dev) if gather else None
        _lib.check(lib.frr_nms_sorted(boxes.data_ptr(), _ptr(counts), B, n, float(iou_threshold), mk, keep.data_ptr(),
                                      cnt.data_ptr(), _ptr(rois), int(cluster_size), int(threads), int(first_chunk),
                                      int(max_chunk), int(lanes_screen), int(lanes_pairs), int(bool(unit_boxes)), _stream()),
                   "frr_nms_sorted")
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
def _feat_layout(feat: torch.Tensor, name: str = "features", shape=(None, None, None, None), device=None):
    """Checks a CUDA fp32 [B,C,H,W] map (of ``shape``, on ``device``: see ``_check``) and returns (tensor usable in place,
    channels_last flag).  NCHW-contiguous and channels_last memory are both consumed without a copy; anything else is
    made NCHW-contiguous."""
    _check(feat, name, torch.float32, shape, device)
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


def rois5(rois, count, feat_hw, out=None, image_hw=None, stride: int = 16):
    """models/model.py:104-110 for a batch: normalised rois [B,R,4] (+ int32 count [B] or None) -> [B*R,5] feature-map
    rois with the batch index; rows past count[b] are masked (index -1).  One kernel, no host synchronisation.
    ``image_hw`` [B,2] (mixed-size batch, ``feat_hw`` = the padded grid): image b is scaled by its own grid
    (W_b // stride, H_b // stride)."""
    lib = _lib.load()
    rois = _req(rois, "rois", shape=(None, None, 4))
    B, R, dev = rois.shape[0], rois.shape[1], rois.device
    if count is not None:
        count = _req(count, "count", torch.int32, (B,), dev)
    if out is not None:
        _check(out, "out", shape=(B * R, 5), device=dev, contiguous=True)
    with torch.cuda.device(dev):
        if out is None:
            out = torch.empty((B * R, 5), dtype=torch.float32, device=dev)
        hw = None if image_hw is None else sized_hw(image_hw, B, feat_hw, stride, dev)
        _lib.check(lib.frr_rois5(rois.data_ptr(), _ptr(count), B, R, int(feat_hw[0]), int(feat_hw[1]), _ptr(hw), int(stride),
                                 out.data_ptr(), _stream()), "frr_rois5")
    return out


def roi_pool_forward(feat, rois5, output_size=(7, 7), spatial_scale: float = 1.0, want_argmax: bool = True,
                     image_hw=None, stride: int = 16):
    """``image_hw`` [B,2] (mixed-size batch padded to the map's H x W cells): every bin window of a roi of image b is
    clipped to that image's own grid (H_b // stride, W_b // stride) -- stride 1 when ``image_hw`` holds feature extents."""
    lib = _lib.load()
    feat, cl = _feat_layout(feat)
    (B, C, H, W), dev = feat.shape, feat.device
    rois5 = _req(rois5, "rois", shape=(None, 5), device=dev)
    K = rois5.shape[0]
    PH, PW = int(output_size[0]), int(output_size[1])
    with torch.cuda.device(dev):
        out = torch.empty((K, C, PH, PW), dtype=torch.float32, device=dev)
        arg = torch.empty((K, C, PH, PW), dtype=torch.int32, device=dev) if want_argmax else None
        hw = None if image_hw is None else sized_hw(image_hw, B, (H, W), stride, dev)
        _lib.check(lib.frr_roi_pool_fwd(feat.data_ptr(), rois5.data_ptr(), K, B, C, H, W, PH, PW, float(spatial_scale), cl,
                                        _ptr(hw), int(stride), out.data_ptr(), _ptr(arg), _stream()), "frr_roi_pool_fwd")
    return out, arg


def _deterministic(flag):
    return torch.are_deterministic_algorithms_enabled() if flag is None else bool(flag)


def roi_pool_backward(grad_out, argmax, rois5, feat_shape, spatial_scale: float = 1.0, channels_last: bool = False,
                      deterministic: bool | None = None, image_hw=None, stride: int = 16):
    """``deterministic``: True runs the kernel whose gradient is bit-exact with torchvision's CPU backward and the same
    on every run; None (default) follows ``torch.use_deterministic_algorithms``.  ``image_hw``: the per-image sizes the
    forward clipped with (mixed-size batch); the default backward follows argmax and needs none, the deterministic one
    clips each bin window to the image's own grid.  The padding region of the gradient is zero either way."""
    lib = _lib.load()
    det = _deterministic(deterministic)
    B, C, H, W = feat_shape
    rois5 = _req(rois5, "rois", shape=(None, 5))
    K, dev = rois5.shape[0], rois5.device
    grad_out = _req(grad_out, "grad_out", shape=(K, C, None, None), device=dev)
    PH, PW = grad_out.shape[2], grad_out.shape[3]
    argmax = _req(argmax, "argmax", torch.int32, (K, C, PH, PW), dev)
    with torch.cuda.device(dev):
        gin = torch.empty((B, C, H, W), dtype=torch.float32, device=dev,
                          memory_format=torch.channels_last if channels_last else torch.contiguous_format)
        args = (grad_out.data_ptr(), argmax.data_ptr(), rois5.data_ptr(), K, B, C, H, W, PH, PW, float(spatial_scale),
                int(channels_last))
        if det:
            hw = None if image_hw is None else sized_hw(image_hw, B, (H, W), stride, dev)
            _lib.check(lib.frr_roi_pool_bwd_deterministic(*args, _ptr(hw), int(stride), gin.data_ptr(), _stream()),
                       "frr_roi_pool_bwd_deterministic")
        else:
            _lib.check(lib.frr_roi_pool_bwd(*args, gin.data_ptr(), _stream()), "frr_roi_pool_bwd")
    return gin


def roi_align_forward(feat, rois5, output_size=(7, 7), spatial_scale: float = 1.0, sampling_ratio: int = 2,
                      aligned: bool = False, out=None):
    """``out``: write into an existing [K,C,PH,PW] tensor (rows of rois with a negative batch index are left untouched)."""
    lib = _lib.load()
    feat, cl = _feat_layout(feat)
    (B, C, H, W), dev = feat.shape, feat.device
    rois5 = _req(rois5, "rois", shape=(None, 5), device=dev)
    K = rois5.shape[0]
    PH, PW = int(output_size[0]), int(output_size[1])
    if out is not None:
        _check(out, "out", shape=(K, C, PH, PW), device=dev, contiguous=True)
    with torch.cuda.device(dev):
        if out is None:
            out = torch.empty((K, C, PH, PW), dtype=torch.float32, device=dev)
        _lib.check(lib.frr_roi_align_fwd(feat.data_ptr(), rois5.data_ptr(), K, B, C, H, W, PH, PW, float(spatial_scale),
                                         int(sampling_ratio), int(aligned), cl, out.data_ptr(), _stream()),
                   "frr_roi_align_fwd")
    return out


def roi_align_backward(grad_out, rois5, feat_shape, spatial_scale: float = 1.0, sampling_ratio: int = 2,
                       aligned: bool = False, channels_last: bool = False, deterministic: bool | None = None):
    """``deterministic``: as for ``roi_pool_backward``."""
    lib = _lib.load()
    fn = lib.frr_roi_align_bwd_deterministic if _deterministic(deterministic) else lib.frr_roi_align_bwd
    B, C, H, W = feat_shape
    rois5 = _req(rois5, "rois", shape=(None, 5))
    K, dev = rois5.shape[0], rois5.device
    grad_out = _req(grad_out, "grad_out", shape=(K, C, None, None), device=dev)
    PH, PW = grad_out.shape[2], grad_out.shape[3]
    with torch.cuda.device(dev):
        gin = torch.empty((B, C, H, W), dtype=torch.float32, device=dev,
                          memory_format=torch.channels_last if channels_last else torch.contiguous_format)
        _lib.check(fn(grad_out.data_ptr(), rois5.data_ptr(), K, B, C, H, W, PH, PW, float(spatial_scale),
                      int(sampling_ratio), int(aligned), int(channels_last), gin.data_ptr(), _stream()), fn.__name__)
    return gin


class _RoIPoolFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, rois5, output_size, spatial_scale, image_hw, stride):
        feat_l, cl = _feat_layout(feat)
        if image_hw is not None:
            image_hw = sized_hw(image_hw, feat.shape[0], feat.shape[2:], stride, feat.device)
        out, arg = roi_pool_forward(feat_l, rois5, output_size, spatial_scale, want_argmax=True, image_hw=image_hw,
                                    stride=stride)
        ctx.save_for_backward(rois5, arg, image_hw)
        ctx.meta = (tuple(feat.shape), float(spatial_scale), bool(cl), int(stride))
        return out

    @staticmethod
    def backward(ctx, grad_out):
        rois5, arg, image_hw = ctx.saved_tensors
        shape, scale, cl, stride = ctx.meta
        return (roi_pool_backward(grad_out.contiguous(), arg, rois5, shape, scale, cl, image_hw=image_hw, stride=stride),
                None, None, None, None, None)


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


def roi_pool(input, boxes, output_size, spatial_scale: float = 1.0, image_hw=None, stride: int = 16):
    """Drop-in for torchvision.ops.roi_pool (differentiable w.r.t. ``input``).  ``image_hw`` [B,2]: a mixed-size batch
    padded to the map's size; windows are clipped to each image's own grid (see ``roi_pool_forward``), in the forward
    and in the deterministic backward."""
    if isinstance(output_size, int):
        output_size = (output_size, output_size)
    rois5 = convert_rois(boxes, input.device).to(torch.float32)
    return _RoIPoolFn.apply(input, rois5.contiguous(), tuple(output_size), float(spatial_scale), image_hw, int(stride))


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
                       variant: str = "vgg", grid_hw=None):
    """``image_hw`` [B,2] + ``grid_hw`` (mixed-size batch, N = grid_h * grid_w * A): each image's anchors and inside-image
    test are its own, its padding cells are labelled like anchors outside the image."""
    lib = _lib.load()
    eps, inside_only, tie_inclusive = VARIANTS[variant]
    gt = _req(gt, "gt", shape=(None, None, 4))
    B, G, dev = gt.shape[0], gt.shape[1], gt.device
    if G == 0:
        raise IndexError("max(): Expected reduction dim 1 to have non-zero size")   # models/model.py:199
    if gt_count is not None:
        gt_count = _req(gt_count, "gt_count", torch.int32, (B,), dev)
    keep, tptr, A = _table_arg(table)
    hw = None
    if is_sized(image_hw):
        if anchors is not None or grid_hw is None:
            raise ValueError("rpn_targets_assign: per-image sizes need grid_hw and generated anchors")
        hw = sized_hw(image_hw, B, grid_hw, stride, dev)
        H, W = int(grid_hw[0]) * stride, int(grid_hw[1]) * stride      # with hw set: the padded size in pixels
    elif anchors is not None:
        anchors = _req(anchors, "anchors", shape=(N, 4), device=dev)
        H = W = 0
    else:
        H, W = int(image_hw[0]), int(image_hw[1])
    with torch.cuda.device(dev):
        ws = dict(iou_max=torch.empty((B, N), dtype=torch.float32, device=dev),
                  argmax=torch.empty((B, N), dtype=torch.int32, device=dev),
                  label8=torch.empty((B, N), dtype=torch.int8, device=dev),
                  pos_list=torch.empty((B, N), dtype=torch.int32, device=dev),
                  neg_list=torch.empty((B, N), dtype=torch.int32, device=dev),
                  counts=torch.empty((B, 2), dtype=torch.int32, device=dev))
        outs = (ws["iou_max"].data_ptr(), ws["argmax"].data_ptr(), ws["label8"].data_ptr(), ws["pos_list"].data_ptr(),
                ws["neg_list"].data_ptr(), ws["counts"].data_ptr(), _stream())
        thr = (float(np.float32(neg_thr)), float(np.float32(pos_thr)), eps, inside_only, tie_inclusive)
        _lib.check(lib.frr_rpn_targets_assign(gt.data_ptr(), _ptr(gt_count), B, G, _ptr(anchors), tptr, A, H, W, _ptr(hw),
                                              stride, N, *thr, *outs), "frr_rpn_targets_assign")
    ws.update(gt=gt, anchors=anchors, geom=(H, W, stride, table, N), image_hw=hw)
    return ws


def rpn_targets_finalize(ws, disable=None, disable_off=None):
    lib = _lib.load()
    H, W, stride, table, N = ws["geom"]
    keep, tptr, A = _table_arg(table)
    gt = _req(ws["gt"], "ws['gt']", shape=(None, None, 4))
    B, G, dev = gt.shape[0], gt.shape[1], gt.device
    anchors, hw = ws["anchors"], ws["image_hw"]
    if anchors is not None:
        anchors = _req(anchors, "ws['anchors']", shape=(N, 4), device=dev)
    if hw is not None:
        hw = _req(hw, "ws['image_hw']", torch.int32, (B, 2), dev)
    argmax = _req(ws["argmax"], "ws['argmax']", torch.int32, (B, N), dev)
    label8 = _check(ws["label8"], "ws['label8']", torch.int8, (B, N), dev, contiguous=True)
    pos_list = _req(ws["pos_list"], "ws['pos_list']", torch.int32, (B, N), dev)
    neg_list = _req(ws["neg_list"], "ws['neg_list']", torch.int32, (B, N), dev)
    if disable is not None or disable_off is not None:
        disable = _req(disable, "disable", torch.int32, (None,), dev)
        disable_off = _req(disable_off, "disable_off", torch.int32, (3 * B,), dev)
    with torch.cuda.device(dev):
        labels = torch.empty((B, N), dtype=torch.int64, device=dev)
        reg = torch.empty((B, N, 4), dtype=torch.float32, device=dev)
        rest = (argmax.data_ptr(), label8.data_ptr(), pos_list.data_ptr(), neg_list.data_ptr(), _ptr(disable),
                _ptr(disable_off), labels.data_ptr(), reg.data_ptr(), _stream())
        _lib.check(lib.frr_rpn_targets_finalize(gt.data_ptr(), B, G, _ptr(anchors), tptr, A, H, W, _ptr(hw), stride, N,
                                                *rest), "frr_rpn_targets_finalize")
    return labels, reg


def frcnn_targets_assign(rois, roi_count, gt, gt_count, fg_thr=0.5, variant: str = "vgg"):
    lib = _lib.load()
    eps = VARIANTS[variant][0]
    rois = _req(rois, "rois", shape=(None, None, 4))
    B, R, dev = rois.shape[0], rois.shape[1], rois.device
    gt = _req(gt, "gt", shape=(B, None, 4), device=dev)
    G = gt.shape[1]
    if G == 0:
        raise IndexError("max(): Expected reduction dim 1 to have non-zero size")
    if roi_count is not None:
        roi_count = _req(roi_count, "roi_count", torch.int32, (B,), dev)
    if gt_count is not None:
        gt_count = _req(gt_count, "gt_count", torch.int32, (B,), dev)
    M = R + G
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
    rois = _req(ws["rois"], "ws['rois']", shape=(None, None, 4))
    B, R, dev = rois.shape[0], rois.shape[1], rois.device
    gt = _req(ws["gt"], "ws['gt']", shape=(B, None, 4), device=dev)
    G = gt.shape[1]
    roi_count = ws["roi_count"]
    if roi_count is not None:
        roi_count = _req(roi_count, "ws['roi_count']", torch.int32, (B,), dev)
    argmax = _req(ws["argmax"], "ws['argmax']", torch.int32, (B, R + G), dev)
    pos_list = _req(ws["pos_list"], "ws['pos_list']", torch.int32, (B, R + G), dev)
    neg_list = _req(ws["neg_list"], "ws['neg_list']", torch.int32, (B, R + G), dev)
    gt_label = _req(gt_label, "gt_label", torch.int64, (B, G), dev)
    sel = _req(sel, "sel", torch.int32, (B, None), dev)
    S = sel.shape[1]
    sel_n = _req(sel_n, "sel_n", torch.int32, (B, 2), dev)
    std = np.ascontiguousarray(std, dtype=np.float32)
    with torch.cuda.device(dev):
        cls = torch.empty((B, S), dtype=torch.int64, device=dev)
        reg = torch.empty((B, S, 4), dtype=torch.float32, device=dev)
        srois = torch.empty((B, S, 4), dtype=torch.float32, device=dev)
        kidx = torch.empty((B, S), dtype=torch.int32, device=dev)
        _lib.check(lib.frr_frcnn_targets_finalize(rois.data_ptr(), _ptr(roi_count), B, R, gt.data_ptr(),
                                                  gt_label.data_ptr(), G, argmax.data_ptr(), pos_list.data_ptr(),
                                                  neg_list.data_ptr(), sel.data_ptr(), sel_n.data_ptr(), S,
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
    mt_state = _check(mt_state, "mt_state", torch.int32, (626,), contiguous=True)       # advanced in place
    dev, B, N = mt_state.device, None, 0
    rpn_counts = frcnn_counts = label8 = pos_list = neg_list = None
    if ws_rpn is not None:
        rpn_counts = _req(ws_rpn["counts"], "ws_rpn['counts']", torch.int32, (None, 2), dev)
        B = rpn_counts.shape[0]
        label8 = _check(ws_rpn["label8"], "ws_rpn['label8']", torch.int8, (B, None), dev, contiguous=True)   # edited in place
        N = label8.shape[1]
        pos_list = _req(ws_rpn["pos_list"], "ws_rpn['pos_list']", torch.int32, (B, N), dev)
        neg_list = _req(ws_rpn["neg_list"], "ws_rpn['neg_list']", torch.int32, (B, N), dev)
    if ws_frcnn is not None:
        frcnn_counts = _req(ws_frcnn["counts"], "ws_frcnn['counts']", torch.int32, (B, 2), dev)     # the same B
        B = frcnn_counts.shape[0]
    S = max(rpn_batch if ws_rpn is not None else 0, frcnn_batch if ws_frcnn is not None else 0)
    with torch.cuda.device(dev):
        jobs = torch.empty((B, 4, 4), dtype=torch.int32, device=dev)
        draws = torch.empty((B, 4, S), dtype=torch.int32, device=dev)
        sel = sel_n = None
        if ws_frcnn is not None:
            sel = torch.zeros((B, frcnn_batch), dtype=torch.int32, device=dev)
            sel_n = torch.zeros((B, 2), dtype=torch.int32, device=dev)
        _lib.check(lib.frr_sample_targets(_ptr(rpn_counts), _ptr(frcnn_counts), B, int(rpn_batch), int(rpn_max_pos),
                                          int(frcnn_batch), int(frcnn_max_pos), mt_state.data_ptr(), N, _ptr(label8),
                                          _ptr(pos_list), _ptr(neg_list), _ptr(sel), _ptr(sel_n), int(frcnn_batch),
                                          jobs.data_ptr(), draws.data_ptr(), S, _stream()), "frr_sample_targets")
    return sel, sel_n


# ------------------------------------------------------------------------------------------------
# loss side (losses/loss.py:5-59 + the class-row gather of models/model.py:340-341)
# ------------------------------------------------------------------------------------------------
RPN_BETA, FRCNN_BETA = float(np.float32(1 / 9)), 1.0      # losses/loss.py:21,47


def region_loss_kernel(rpn_cls, rpn_reg, frc_cls, frc_reg, rpn_tcls, rpn_treg, frc_tcls, frc_treg, need):
    """One ``frr_region_loss`` launch on arguments checked by ``region_loss_args``: returns loss [B,5] and, for each of
    the four predictions with ``need[j]`` set, the gradient of its image's total for a unit upstream gradient (else
    None)."""
    lib = _lib.load()
    have_rpn, have_frc = rpn_cls is not None, frc_cls is not None
    ref = rpn_cls if have_rpn else frc_cls
    dev = ref.device
    B = ref.shape[0]
    N = rpn_cls.shape[1] if have_rpn else 0
    S, C = (frc_cls.shape[1], frc_cls.shape[2]) if have_frc else (0, 0)
    CR = frc_reg.shape[2] if have_frc else 0
    need = [have_rpn and need[0], have_rpn and need[1], have_frc and need[2], have_frc and need[3]]
    with torch.cuda.device(dev):
        loss = torch.empty((B, 5), dtype=torch.float32, device=dev)
        grads = [torch.empty_like(t) if n else None for t, n in zip((rpn_cls, rpn_reg, frc_cls, frc_reg), need)]
        _lib.check(lib.frr_region_loss(_ptr(rpn_cls), _ptr(rpn_reg), _ptr(rpn_tcls), _ptr(rpn_treg), B, N, _ptr(frc_cls),
                                       _ptr(frc_reg), _ptr(frc_tcls), _ptr(frc_treg), S, C, CR, RPN_BETA, FRCNN_BETA,
                                       loss.data_ptr(), _ptr(grads[0]), _ptr(grads[1]), _ptr(grads[2]), _ptr(grads[3]),
                                       _stream()), "frr_region_loss")
    return loss, grads


def region_loss_scale(saved, g):
    """Gradients of the four predictions for the upstream ``g`` [B,5] of (total, rpn_cls, rpn_reg, frcnn_cls,
    frcnn_reg), from the unit gradients ``region_loss_kernel`` saved (None stays None)."""
    out = []
    for j, s in enumerate(saved):
        if s is None:
            out.append(None)
            continue
        up = (g[:, 0] + g[:, 1 + j]).reshape((-1,) + (1,) * (s.dim() - 1))
        out.append(s * up)
    return out


class _RegionLossFn(torch.autograd.Function):
    """One kernel computes the four losses and, for a unit upstream gradient, their gradients w.r.t. the predictions;
    backward only scales the saved gradients by the upstream values."""

    @staticmethod
    def forward(ctx, rpn_cls, rpn_reg, frc_cls, frc_reg, rpn_tcls, rpn_treg, frc_tcls, frc_treg):
        loss, ctx.grads = region_loss_kernel(rpn_cls, rpn_reg, frc_cls, frc_reg, rpn_tcls, rpn_treg, frc_tcls, frc_treg,
                                             ctx.needs_input_grad[:4])
        return loss

    @staticmethod
    def backward(ctx, g):            # g [B,5]: upstream of (total, rpn_cls, rpn_reg, frcnn_cls, frcnn_reg)
        return tuple(region_loss_scale(ctx.grads, g)) + (None, None, None, None)


def region_loss_args(rpn_cls=None, rpn_reg=None, rpn_target_cls=None, rpn_target_reg=None, frcnn_cls=None, frcnn_reg=None,
                     frcnn_target_cls=None, frcnn_target_reg=None):
    """The checks of ``region_loss``: returns its tensors contiguous, frcnn_reg as [B,S,C|1,4], in the kernel's order
    (rpn_cls, rpn_reg, frcnn_cls, frcnn_reg, rpn_target_cls, rpn_target_reg, frcnn_target_cls, frcnn_target_reg)."""
    if rpn_cls is None and frcnn_cls is None:
        raise ValueError("region_loss: nothing to compute")
    B = dev = None                                        # taken from the RPN half, when given, for both halves
    if rpn_cls is not None:
        rpn_cls = _req(rpn_cls, "rpn_cls", shape=(None, None, 2))
        B, N, dev = rpn_cls.shape[0], rpn_cls.shape[1], rpn_cls.device
        rpn_reg = _req(rpn_reg, "rpn_reg", shape=(B, N, 4), device=dev)
        rpn_target_cls = _req(rpn_target_cls, "rpn_target_cls", torch.int64, (B, N), dev)
        rpn_target_reg = _req(rpn_target_reg, "rpn_target_reg", shape=(B, N, 4), device=dev)
    if frcnn_cls is not None:
        frcnn_cls = _req(frcnn_cls, "frcnn_cls", shape=(B, None, None), device=dev)
        (B, S, C), dev = frcnn_cls.shape, frcnn_cls.device
        frcnn_reg = _req(frcnn_reg, "frcnn_reg", device=dev)
        if frcnn_reg.numel() == B * S * C * 4:
            frcnn_reg = frcnn_reg.reshape(B, S, C, 4)
        elif frcnn_reg.numel() == B * S * 4:
            frcnn_reg = frcnn_reg.reshape(B, S, 1, 4)
        else:
            raise ValueError("region_loss: frcnn_reg must hold C or 1 rows of 4 per sample")
        frcnn_target_cls = _req(frcnn_target_cls, "frcnn_target_cls", torch.int64, (B, S), dev)
        frcnn_target_reg = _req(frcnn_target_reg, "frcnn_target_reg", shape=(B, S, 4), device=dev)
    return rpn_cls, rpn_reg, frcnn_cls, frcnn_reg, rpn_target_cls, rpn_target_reg, frcnn_target_cls, frcnn_target_reg


def region_loss(rpn_cls=None, rpn_reg=None, rpn_target_cls=None, rpn_target_reg=None, frcnn_cls=None, frcnn_reg=None,
                frcnn_target_cls=None, frcnn_target_reg=None):
    """Batched FRCNNLoss (losses/loss.py:62-82): per image (total, rpn_cls, rpn_reg, frcnn_cls, frcnn_reg) -> [B,5],
    differentiable w.r.t. the four prediction tensors.  rpn_cls [B,N,2], rpn_reg [B,N,4], rpn_target_cls int64 [B,N],
    rpn_target_reg [B,N,4]; frcnn_cls [B,S,C], frcnn_reg [B,S,C,4] (or [B,S,C*4]: the head output, the class row is
    gathered in the kernel, models/model.py:340-341) or [B,S,4] (already gathered), frcnn_target_cls int64 [B,S]
    (negative = padding), frcnn_target_reg [B,S,4].  Either half may be omitted."""
    return _RegionLossFn.apply(*region_loss_args(rpn_cls, rpn_reg, rpn_target_cls, rpn_target_reg, frcnn_cls, frcnn_reg,
                                                 frcnn_target_cls, frcnn_target_reg))


# ------------------------------------------------------------------------------------------------
# detection post-processing (D1, D2)
# ------------------------------------------------------------------------------------------------
def decode_classwise(cls_logits, reg, rois, num_classes: int, std=_STD4):
    """cls [rows,C], reg [rows,4C], rois [rows,4] -> prob [rows,C], boxes [rows,4C] (clamped to [0,1])."""
    lib = _lib.load()
    C = int(num_classes)
    cls_logits = _req(cls_logits, "cls_logits", shape=(None, C))
    rows, dev = cls_logits.shape[0], cls_logits.device
    rois = _req(rois, "rois", shape=(rows, 4), device=dev)
    reg = _req(reg, "reg", device=dev)
    if reg.numel() != rows * C * 4:
        raise ValueError(f"decode_classwise: reg must hold {C} rows of 4 per roi ([rows,{4 * C}] or [rows,{C},4])")
    std = np.ascontiguousarray(std, dtype=np.float32)
    with torch.cuda.device(dev):
        prob = torch.empty((rows, C), dtype=torch.float32, device=dev)
        boxes = torch.empty((rows, C * 4), dtype=torch.float32, device=dev)
        _lib.check(lib.frr_decode_classwise(cls_logits.data_ptr(), reg.data_ptr(), rois.data_ptr(), rows, C, std.ctypes.data,
                                            prob.data_ptr(), boxes.data_ptr(), _stream()), "frr_decode_classwise")
    return prob, boxes


def class_nms(prob, boxes, num_classes: int, score_thres: float = 0.05, iou_thr: float = 0.3, roi_count=None, cap=None):
    """prob [B,R,C], boxes [B,R,4C] -> det_boxes [B,cap,4], det_labels int32 [B,cap], det_scores [B,cap], count [B]."""
    lib = _lib.load()
    C = int(num_classes)
    prob = _req(prob, "prob", shape=(None, None, C))
    B, R, dev = prob.shape[0], prob.shape[1], prob.device
    boxes = _req(boxes, "boxes", device=dev)
    if boxes.numel() != B * R * C * 4:
        raise ValueError(f"class_nms: boxes must hold {C} boxes per roi ([B,R,{4 * C}] or [B,R,{C},4])")
    if roi_count is not None:
        roi_count = _req(roi_count, "roi_count", torch.int32, (B,), dev)
    cap = R * (C - 1) if cap is None else int(cap)
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


def check_rank(rank: str, per_class_max: int):
    """Raises ValueError unless (rank, per_class_max) is a selection ``pack_detections`` offers."""
    if rank not in ("class", "score"):
        raise ValueError(f"pack_detections: rank must be 'class' or 'score', got {rank!r}")
    if int(per_class_max) < 0 or (rank == "class" and int(per_class_max) != 0):
        raise ValueError("pack_detections: per_class_max is a count >= 0 and applies to rank='score' only")


def pack_ranked_workspace(B: int, cap: int, max_det: int, device) -> torch.Tensor:
    """Workspace of ``pack_detections(..., rank="score")`` for ``[B,cap]`` detections and ``max_det`` rows: allocate it
    once and pass it to every call (a captured CUDA graph then allocates nothing for the ranking)."""
    nbytes = int(_lib.load().frr_pack_detections_ranked_workspace_bytes(int(B), int(cap), int(max_det)))
    return torch.empty((nbytes + 256,), dtype=torch.uint8, device=device)


def pack_detections(det_boxes, det_labels, det_scores, det_count, max_det: int, image_wh=None, xywh: bool = False,
                    rank: str = "class", per_class_max: int = 0, workspace=None):
    """Evaluation hand-off (test.py:68-88, evaluation/coco_eval.py:156-158): [B,cap,4] / [B,cap] / [B,cap] / [B] ->
    ([B,max_det,6] rows (x, y, x2|w, y2|h, score, label) scaled by ``image_wh [B,2]`` = (w, h), int32 counts [B]).

    Which ``max_det`` detections of an image become its rows (the input is ``class_nms``'s class-major output):
    ``rank="class"`` keeps the first ``max_det`` in class order; ``rank="score"`` keeps the ``max_det`` highest scores
    (ties: lower class-major position first), after dropping, with ``per_class_max > 0``, every detection past the
    first ``per_class_max`` of its class.  ``rank="score", max_det=100`` is the torchvision / Detectron per-image cap;
    ``per_class_max=100`` with a large ``max_det`` hands COCOeval (maxDets 100) every detection it can score.  The
    ranking sees only the rows ``class_nms`` kept: leave its ``cap`` at the default ``R*(C-1)`` for a complete one.
    ``workspace``: from ``pack_ranked_workspace`` (allocated here when None)."""
    check_rank(rank, per_class_max)
    lib = _lib.load()
    det_labels = _req(det_labels, "det_labels", torch.int32, (None, None))
    (B, cap), dev = det_labels.shape, det_labels.device
    det_boxes = _req(det_boxes, "det_boxes", shape=(B, cap, 4), device=dev)
    det_scores = _req(det_scores, "det_scores", shape=(B, cap), device=dev)
    det_count = _req(det_count, "det_count", torch.int32, (B,), dev)
    if image_wh is not None:
        image_wh = _req(image_wh, "image_wh", shape=(B, 2), device=dev)
    if workspace is not None:
        workspace = _req(workspace, "workspace", torch.uint8, device=dev)
    with torch.cuda.device(dev):
        out = torch.empty((B, int(max_det), 6), dtype=torch.float32, device=dev)
        cnt = torch.empty((B,), dtype=torch.int32, device=dev)
        if rank == "class":
            _lib.check(lib.frr_pack_detections(det_boxes.data_ptr(), det_labels.data_ptr(), det_scores.data_ptr(),
                                               det_count.data_ptr(), B, cap, int(max_det), _ptr(image_wh), int(bool(xywh)),
                                               out.data_ptr(), cnt.data_ptr(), _stream()), "frr_pack_detections")
            return out, cnt
        if workspace is None:
            workspace = pack_ranked_workspace(B, cap, max_det, dev)
        off = (-workspace.data_ptr()) % 256
        _lib.check(lib.frr_pack_detections_ranked(det_boxes.data_ptr(), det_labels.data_ptr(), det_scores.data_ptr(),
                                                  det_count.data_ptr(), B, cap, int(max_det), int(per_class_max),
                                                  _ptr(image_wh), int(bool(xywh)), out.data_ptr(), cnt.data_ptr(),
                                                  workspace.data_ptr() + off, max(workspace.numel() - off, 0), _stream()),
                   "frr_pack_detections_ranked")
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
    rois5 = _req(rois5, "rois", shape=(None, 5))
    K, L, dev = rois5.shape[0], k_max - k_min + 1, rois5.device
    with torch.cuda.device(dev):
        levels = torch.empty((K,), dtype=torch.int32, device=dev)
        per = torch.empty((L, K, 5), dtype=torch.float32, device=dev)
        _lib.check(lib.frr_fpn_level_rois(rois5.data_ptr(), K, int(k_min), int(k_max), int(canonical_level),
                                          float(canonical_scale), L, levels.data_ptr(), per.data_ptr(), _stream()),
                   "frr_fpn_level_rois")
    return levels, per


def multiscale_roi_align_forward(feats, rois5, output_size, sampling_ratio: int, scales, k_min: int, k_max: int,
                                 canonical_scale: float = 224.0, canonical_level: int = 4):
    """The kernels of ``multiscale_roi_align`` for given per-level ``scales`` (see ``infer_scales``): returns (out
    [K,C,PH,PW], levels int32 [K], the per-level rois [L,K,5] the backward reads, channels_last flag per level)."""
    if len(feats) != k_max - k_min + 1:
        raise ValueError(f"multiscale_roi_align: one feature map per level {k_min}..{k_max}, got {len(feats)} maps")
    maps = [_feat_layout(feats[0], "features[0]")]
    C, dev = maps[0][0].shape[1], maps[0][0].device
    maps += [_feat_layout(f, f"features[{l}]", (None, C, None, None), dev) for l, f in enumerate(feats[1:], 1)]
    rois5 = _req(rois5, "rois", shape=(None, 5), device=dev)
    levels, per = fpn_level_rois(rois5, k_min, k_max, canonical_scale, canonical_level)
    out = torch.empty((rois5.shape[0], C, output_size[0], output_size[1]), dtype=torch.float32, device=dev)
    for l, (f_l, _) in enumerate(maps):
        roi_align_forward(f_l, per[l], output_size, scales[l], sampling_ratio, False, out=out)
    return out, levels, per, [bool(cl) for _, cl in maps]


def multiscale_roi_align_backward(grad_out, per, shapes, scales, sampling_ratio: int, lay):
    """Feature gradients (one per level, [B,C,Hl,Wl], channels_last where ``lay[l]``) of ``multiscale_roi_align_forward``."""
    go = grad_out.contiguous()
    return [roi_align_backward(go, per[l], shapes[l], scales[l], sampling_ratio, False, lay[l]) for l in range(len(shapes))]


class _MultiScaleRoIAlignFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rois5, output_size, sampling_ratio, scales, k_min, k_max, canonical_scale, canonical_level, *feats):
        out, levels, per, lay = multiscale_roi_align_forward(feats, rois5, output_size, sampling_ratio, scales, k_min, k_max,
                                                             canonical_scale, canonical_level)
        ctx.save_for_backward(per)
        ctx.meta = ([tuple(f.shape) for f in feats], list(scales), int(sampling_ratio), lay)
        ctx.mark_non_differentiable(levels)
        return out, levels

    @staticmethod
    def backward(ctx, grad_out, _grad_levels):
        (per,) = ctx.saved_tensors
        shapes, scales, sr, lay = ctx.meta
        return (None,) * 8 + tuple(multiscale_roi_align_backward(grad_out, per, shapes, scales, sr, lay))


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
