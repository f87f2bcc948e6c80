"""Host side of the target makers: the reference's sampling logic around the assign/finalize kernels.

The reference draws its samples with ``torch.randperm`` on the host generator and the number and length of
the draws depend on the data (models/model.py:225-236,147-156).  Two ways to reproduce the sampled indices bit for
bit under ``torch.manual_seed``:

* host sampling (default, ``generator=None``): the permutations are drawn here with ``torch.randperm`` in the
  reference's order; the device needs ONE small D2H copy of the candidate counts per batch (the reference syncs
  >= 5 times per image);
* device sampling (``generator=DeviceGenerator(...)``): torch's mt19937 state is copied to the device once and the
  draws are replayed there (``frr_sample_targets``) -- no synchronisation at all; ``DeviceGenerator.sync_to_torch()``
  hands the advanced state back when something else needs the host generator.
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops

RPN_BATCH, RPN_MAX_POS = 256, 128            # models/model.py:225-236
FRCNN_BATCH, FRCNN_MAX_POS = 128, 32         # models/model.py:144,151


_MT_N = 624
_ST_LEFT, _ST_NEXT, _ST_WORDS = 8, 16, 24        # byte offsets in torch's CPU generator state (legacy mt19937 POD)


class DeviceGenerator:
    """torch's CPU mt19937 generator, resident on the device.  ``state`` int32 [626]: the 624 state words, the index of
    the next unread word (624 = exhausted), one reserved word.  Created from the default CPU generator (or a given
    ``torch.Generator``) AFTER seeding; as long as nothing else draws from that host generator in between, the device
    draws are exactly the numbers the reference's ``torch.randperm`` calls would have consumed."""

    def __init__(self, device, generator: torch.Generator | None = None):
        self.device = torch.device(device)
        self.generator = generator
        self.state = None
        self.sync_from_torch()

    def _host_state(self):
        return self.generator.get_state() if self.generator is not None else torch.get_rng_state()

    def sync_from_torch(self):
        raw = self._host_state().numpy()
        left = int(raw[_ST_LEFT:_ST_LEFT + 4].view(np.int32)[0])
        nxt = int(raw[_ST_NEXT:_ST_NEXT + 8].view(np.uint64)[0])
        words = raw[_ST_WORDS:_ST_WORDS + 8 * _MT_N].view(np.uint64).astype(np.uint32)
        st = np.zeros((_MT_N + 2,), np.uint32)
        st[:_MT_N] = words
        st[_MT_N] = _MT_N if left == 1 else nxt              # left == 1: the engine twists before its next output
        self.state = torch.from_numpy(st.view(np.int32)).to(self.device)
        return self

    def sync_to_torch(self):
        """Write the advanced state back into the host generator (one D2H copy + synchronisation)."""
        st = self.state.cpu().numpy().view(np.uint32)
        raw = self._host_state().numpy().copy()
        pos = int(st[_MT_N])
        raw[_ST_WORDS:_ST_WORDS + 8 * _MT_N] = st[:_MT_N].astype(np.uint64).view(np.uint8)
        raw[_ST_NEXT:_ST_NEXT + 8] = np.asarray([pos], np.uint64).view(np.uint8)
        raw[_ST_LEFT:_ST_LEFT + 4] = np.asarray([_MT_N + 1 - pos], np.int32).view(np.uint8)
        t = torch.from_numpy(raw)
        if self.generator is not None:
            self.generator.set_state(t)
        else:
            torch.set_rng_state(t)
        return self


def _perm(randperm, n):
    p = randperm(int(n))
    return p.numpy() if isinstance(p, torch.Tensor) else np.asarray(p)


def rpn_disable_positions(n_pos: int, n_neg: int, randperm):
    """models/model.py:225-236: which positions of the ordered positive / negative lists become ignore (-1)."""
    dis_pos = np.zeros((0,), np.int64)
    dis_neg = np.zeros((0,), np.int64)
    if n_pos > RPN_MAX_POS:
        dis_pos = _perm(randperm, n_pos)[RPN_MAX_POS:]
    if n_neg > RPN_BATCH - n_pos:
        if n_pos > RPN_MAX_POS:
            n_pos = RPN_MAX_POS
        dis_neg = _perm(randperm, n_neg)[RPN_BATCH - n_pos:]
    return dis_pos, dis_neg


FRCNN_SAMPLING = {"vgg": (FRCNN_BATCH, FRCNN_MAX_POS), "fpn": (512, 128)}   # models/new_model.py:169-177


def frcnn_select_positions(n_pos_cand: int, n_neg_cand: int, randperm, batch: int = FRCNN_BATCH,
                           max_pos: int = FRCNN_MAX_POS):
    """models/model.py:144-156: both permutations are always drawn; returns (positions, n_pos)."""
    n_pos = int(min(n_pos_cand, max_pos))
    sel_pos = _perm(randperm, n_pos_cand)[:n_pos]
    sel_neg = _perm(randperm, n_neg_cand)[:batch - n_pos]
    return np.concatenate([sel_pos, sel_neg]).astype(np.int32), n_pos


def _upload_disable(per_image, device):
    flat, off = [], []
    run = 0
    for dp, dn in per_image:
        off += [run, run + len(dp), run + len(dp) + len(dn)]
        run += len(dp) + len(dn)
        flat += [dp, dn]
    flat = np.concatenate(flat).astype(np.int32) if run else np.zeros((1,), np.int32)
    return (torch.from_numpy(flat).to(device, non_blocking=True),
            torch.from_numpy(np.asarray(off, dtype=np.int32)).to(device, non_blocking=True))


def _upload_select(per_image, device, batch: int = FRCNN_BATCH):
    B = len(per_image)
    sel = np.zeros((B, batch), np.int32)
    sel_n = np.zeros((B, 2), np.int32)
    for b, (s, n_pos) in enumerate(per_image):
        sel[b, :len(s)] = s
        sel_n[b] = (n_pos, len(s))
    return torch.from_numpy(sel).to(device, non_blocking=True), torch.from_numpy(sel_n).to(device, non_blocking=True)


def _anchor_count(image_hw, anchors, grid_hw):
    if anchors is not None:
        return anchors.shape[0]
    if ops.is_sized(image_hw):
        if grid_hw is None:
            raise ValueError("per-image sizes need grid_hw, the padded grid in cells")
        return int(grid_hw[0]) * int(grid_hw[1]) * 9
    return (image_hw[0] // 16) * (image_hw[1] // 16) * 9


def rpn_targets(gt, gt_count=None, image_hw=None, anchors=None, N=None, randperm=torch.randperm, generator=None,
                grid_hw=None, **kw):
    """Batched RPNTargetMaker: gt [B,Gmax,4] (+ gt_count) -> labels int64 [B,N], reg fp32 [B,N,4].
    ``variant="fpn"`` = models/new_model.py:299-349 (no inside filter, eps-free IoU, tie-inclusive low-quality match).
    ``generator``: a ``DeviceGenerator`` -> sampling on the device, no host synchronisation.
    Mixed-size batch: ``image_hw`` [B,2] per-image sizes and ``grid_hw`` the padded grid in cells; every image gets the
    labels and draws it would get alone, its padding cells label -1 and a zero target."""
    if N is None:
        N = _anchor_count(image_hw, anchors, grid_hw)
    ws = ops.rpn_targets_assign(gt, gt_count, N, image_hw=image_hw, anchors=anchors, grid_hw=grid_hw, **kw)
    if generator is not None:
        ops.sample_targets(generator.state, ws_rpn=ws, rpn_batch=RPN_BATCH, rpn_max_pos=RPN_MAX_POS)
        return ops.rpn_targets_finalize(ws)
    counts = ws["counts"].cpu().numpy()                       # the one host sync
    per_image = [rpn_disable_positions(int(c[0]), int(c[1]), randperm) for c in counts]
    disable, off = _upload_disable(per_image, gt.device)
    return ops.rpn_targets_finalize(ws, disable, off)


def frcnn_targets(rois, roi_count, gt, gt_count, gt_label, randperm=torch.randperm, variant: str = "vgg", generator=None):
    """Batched FastRcnnTargetMaker: -> cls int64 [B,S], reg [B,S,4], sample_rois [B,S,4], n int32 [B] (host); S = 128
    (``variant="vgg"``, models/model.py:127-179) or 512 (``"fpn"``, models/new_model.py:153-206).
    ``generator``: a ``DeviceGenerator`` -> sampling on the device; n is then a device tensor (no synchronisation)."""
    batch, max_pos = FRCNN_SAMPLING[variant]
    ws = ops.frcnn_targets_assign(rois, roi_count, gt, gt_count, variant=variant)
    if generator is not None:
        sel, sel_n = ops.sample_targets(generator.state, ws_frcnn=ws, frcnn_batch=batch, frcnn_max_pos=max_pos)
        cls, reg, srois, kidx = ops.frcnn_targets_finalize(ws, gt_label, sel, sel_n, label_offset=0 if variant == "fpn" else 1)
        return cls, reg, srois, kidx, sel_n[:, 1]
    counts = ws["counts"].cpu().numpy()
    per_image = [frcnn_select_positions(int(c[0]), int(c[1]), randperm, batch, max_pos) for c in counts]
    sel, sel_n = _upload_select(per_image, rois.device, batch)
    cls, reg, srois, kidx = ops.frcnn_targets_finalize(ws, gt_label, sel, sel_n, label_offset=0 if variant == "fpn" else 1)
    return cls, reg, srois, kidx, np.asarray([len(s) for s, _ in per_image], dtype=np.int32)


def make_targets(gt, gt_count, gt_label, rois, roi_count, image_hw=None, anchors=None, N=None, randperm=torch.randperm,
                 generator=None, grid_hw=None):
    """Both target makers for a batch.  Permutations are drawn per image in the reference's order (RPN positives, RPN
    negatives, Fast R-CNN positives, Fast R-CNN negatives): on the host with a single synchronisation (default), or on
    the device with none (``generator`` = a ``DeviceGenerator``; ``n_samples`` is then a device tensor).
    ``image_hw`` [B,2] + ``grid_hw``: a mixed-size batch, as in ``rpn_targets``."""
    if N is None:
        N = _anchor_count(image_hw, anchors, grid_hw)
    ws_r = ops.rpn_targets_assign(gt, gt_count, N, image_hw=image_hw, anchors=anchors, grid_hw=grid_hw)
    ws_f = ops.frcnn_targets_assign(rois, roi_count, gt, gt_count)
    if generator is not None:
        sel, sel_n = ops.sample_targets(generator.state, ws_rpn=ws_r, ws_frcnn=ws_f, rpn_batch=RPN_BATCH,
                                        rpn_max_pos=RPN_MAX_POS, frcnn_batch=FRCNN_BATCH, frcnn_max_pos=FRCNN_MAX_POS)
        labels, reg = ops.rpn_targets_finalize(ws_r)
        cls, freg, srois, kidx = ops.frcnn_targets_finalize(ws_f, gt_label, sel, sel_n)
        return dict(rpn_cls=labels, rpn_reg=reg, frcnn_cls=cls, frcnn_reg=freg, sample_rois=srois, keep_index=kidx,
                    n_samples=sel_n[:, 1])
    counts = torch.cat([ws_r["counts"], ws_f["counts"]], dim=1).cpu().numpy()       # one D2H for the batch
    dis, sels = [], []
    for c in counts:
        dis.append(rpn_disable_positions(int(c[0]), int(c[1]), randperm))
        sels.append(frcnn_select_positions(int(c[2]), int(c[3]), randperm))
    disable, off = _upload_disable(dis, gt.device)
    sel, sel_n = _upload_select(sels, gt.device)
    labels, reg = ops.rpn_targets_finalize(ws_r, disable, off)
    cls, freg, srois, kidx = ops.frcnn_targets_finalize(ws_f, gt_label, sel, sel_n)
    return dict(rpn_cls=labels, rpn_reg=reg, frcnn_cls=cls, frcnn_reg=freg, sample_rois=srois, keep_index=kidx,
                n_samples=np.asarray([len(s) for s, _ in sels], dtype=np.int32))
