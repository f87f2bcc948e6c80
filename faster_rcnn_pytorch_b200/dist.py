"""Multi-GPU plumbing of the region stage: one process per GPU (torch.distributed; NCCL on GPUs, gloo in the
CPU tests).  Images are independent, so the stage shards by image with NO data-path collective
(``shard_range`` = the contiguous split ``DistributedSampler`` style launchers use, main.py:117-121 /
new_datasets/build.py:65-73); the only exchange is the evaluation hand-off, where the reference all-gathers
PICKLED per-rank results (util/misc.py:89-129 via evaluation/coco_eval.py:161-180).  ``gather_detections``
replaces that with one fixed-shape tensor all-gather: [B_local, max_det, 6] fp32 + int32 counts + int64 ids.
"""
from __future__ import annotations

import torch
import torch.distributed as dist


def world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_range(n_items: int, rank: int | None = None, world_size: int | None = None):
    """Contiguous, balanced shard [lo, hi) of ``n_items`` images for ``rank``: the first n % world ranks get one
    extra image.  Every image belongs to exactly one rank."""
    if rank is None or world_size is None:
        rank, world_size = world()
    base, extra = divmod(int(n_items), int(world_size))
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def pack_detections(det_boxes, det_labels, det_scores, det_count, max_det: int, image_wh=None, xywh: bool = False,
                    rank: str = "class", per_class_max: int = 0, workspace=None):
    """[B,cap,4] boxes, [B,cap] int32 labels, [B,cap] scores, [B] counts (class-major order as produced by
    ``ops.class_nms``) -> ([B,max_det,6] fp32 rows (x, y, x2|w, y2|h, score, label), [B] int32 counts): ``max_det``
    detections of every image, rows past the count zero; optional pixel scaling and xyxy -> xywh
    (test.py:68-88, evaluation/coco_eval.py:156-158).  ``rank="class"`` (one ``frr_pack_detections`` kernel) keeps the
    first ``max_det`` in class order, ``rank="score"`` (``frr_pack_detections_ranked``) the highest-scoring ones, at
    most ``per_class_max`` per class when that is > 0: see ``ops.pack_detections``."""
    from . import ops
    return ops.pack_detections(det_boxes, det_labels, det_scores, det_count, max_det, image_wh=image_wh, xywh=xywh,
                               rank=rank, per_class_max=per_class_max, workspace=workspace)


def gather_detections(packed, counts, image_ids, group=None, equal_batch: bool = False):
    """All-gather fixed-shape detections from every rank (one collective per tensor, no pickling, no host copy).
    ``equal_batch=True``: the caller guarantees the same B_local on every rank (the usual sharded-eval case); the size
    exchange and its host synchronisation are skipped and the call is fully asynchronous.

    packed [B_local,max_det,6] fp32, counts [B_local] int32, image_ids [B_local] int64.  Ranks may hold different
    B_local (the last shard can be short): tensors are padded to the largest local batch, padding rows carry
    image id -1 and are dropped.  Returns (packed [B_total,max_det,6], counts [B_total], image_ids [B_total])
    ordered by rank, identical on every rank."""
    rank, ws = world()
    if ws == 1:
        return packed, counts, image_ids
    dev = packed.device
    if equal_batch:
        B = packed.shape[0]
        P = torch.empty((ws * B,) + tuple(packed.shape[1:]), dtype=packed.dtype, device=dev)
        Cn = torch.empty((ws * B,), dtype=torch.int32, device=dev)
        I = torch.empty((ws * B,), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(P, packed.contiguous(), group=group)
        dist.all_gather_into_tensor(Cn, counts.to(torch.int32).contiguous(), group=group)
        dist.all_gather_into_tensor(I, image_ids.to(torch.int64).contiguous(), group=group)
        return P, Cn, I
    b_local = torch.tensor([packed.shape[0]], dtype=torch.int64, device=dev)
    sizes = [torch.zeros_like(b_local) for _ in range(ws)]
    dist.all_gather(sizes, b_local, group=group)
    b_max = int(max(int(s.item()) for s in sizes))

    def pad(t, fill):
        if t.shape[0] == b_max:
            return t.contiguous()
        extra = torch.full((b_max - t.shape[0],) + tuple(t.shape[1:]), fill, dtype=t.dtype, device=dev)
        return torch.cat([t, extra], dim=0).contiguous()

    p, c, i = pad(packed, 0.0), pad(counts.to(torch.int32), 0), pad(image_ids.to(torch.int64), -1)
    gp = [torch.empty_like(p) for _ in range(ws)]
    gc = [torch.empty_like(c) for _ in range(ws)]
    gi = [torch.empty_like(i) for _ in range(ws)]
    dist.all_gather(gp, p, group=group)
    dist.all_gather(gc, c, group=group)
    dist.all_gather(gi, i, group=group)
    P, Cn, I = torch.cat(gp, 0), torch.cat(gc, 0), torch.cat(gi, 0)
    keep = I >= 0
    return P[keep], Cn[keep], I[keep]
