"""Batched region-stage pipelines built from the libfrr kernels (the public functional API).

``rpn_proposals`` is the batched equivalent of the reference's ``RegionProposal.forward``
(models/model.py:17-58): decode+clip+min-size -> top-k -> NMS -> first post_nms boxes, for B images
at once, with no host synchronisation (ragged sizes come back as counts on the device).

``ProposalPlan`` is the same computation with every buffer allocated once and the three kernels
issued by ONE C-ABI call (``frr_rpn_proposals``), so a step costs one ctypes call on the host and is
CUDA-graph capturable.  ``HostProposalPipeline`` wraps a plan for callers whose RPN head outputs live in
host memory: pinned staging, H2D on a copy stream, kernels, D2H of rois + counts, double buffered so the
copies of step i+1 overlap the kernels of step i.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib, ops

PROPOSAL_MODES = {"train": (12000, 2000), "test": (6000, 300)}   # models/model.py:24-28
RPN_NMS_THRESH = 0.7                                              # models/model.py:53


def rpn_head_views(cls_map, reg_map):
    """RPN head hand-off (models/model.py:82-83): ``cls_map [B,2A,H,W]``, ``reg_map [B,4A,H,W]`` (the outputs of the
    two 1x1 convs) -> ``cls [B,H*W*A,2]``, ``reg [B,H*W*A,4]`` in the reference's anchor order.

    The reference does ``permute(0,2,3,1).contiguous().view(B,-1,k)``: a copy of 6N floats per image.  When the convs
    run in ``torch.channels_last`` the permuted tensor IS contiguous and the views below alias the conv outputs
    (zero copy: ``[B,H,W,A*4]`` is ``[B,N,4]``); for NCHW-contiguous maps this falls back to the reference's copy."""
    B = cls_map.shape[0]
    cls = cls_map.permute(0, 2, 3, 1)
    reg = reg_map.permute(0, 2, 3, 1)
    if not cls.is_contiguous():
        cls = cls.contiguous()
    if not reg.is_contiguous():
        reg = reg.contiguous()
    return cls.view(B, -1, 2), reg.view(B, -1, 4)


def rpn_proposals(cls, reg, image_hw=None, mode: str = "train", anchors=None, stride: int = 16, table=None,
                  pre_nms_top_k: int | None = None, post_nms_top_k: int | None = None,
                  nms_thresh: float = RPN_NMS_THRESH, cluster_size: int = 0, return_all: bool = False,
                  min_size: float = ops._MIN_SIZE, grid_hw=None):
    """cls [B,N,2] logits (or [B,N] fg scores), reg [B,N,4] -> rois [B,post,4] (zero padded), count int32 [B].
    ``min_size`` is the normalised side threshold (models/model.py:39: 1/1000; models/new_model.py:66: 10/1000).
    Mixed-size batch: ``image_hw`` [B,2] per-image (H, W) and ``grid_hw`` the padded grid in cells (N = grid_h * grid_w
    * A); every image's proposals are those it gets alone at its own size (top-k indices refer to the padded N)."""
    pre_k, post_k = PROPOSAL_MODES[mode]
    pre_k = pre_k if pre_nms_top_k is None else int(pre_nms_top_k)
    post_k = post_k if post_nms_top_k is None else int(post_nms_top_k)
    boxes, scores, valid = ops.rpn_decode(reg, cls, image_hw=image_hw, anchors=anchors, stride=stride, table=table,
                                          min_size=min_size, grid_hw=grid_hw)
    k = min(pre_k, boxes.shape[1])
    top = ops.topk_desc(scores, k, valid=valid, boxes=boxes, want_cidx=return_all)
    keep, count, rois = ops.nms_sorted(top["boxes"], nms_thresh, max_keep=post_k, counts=top["count"],
                                       cluster_size=cluster_size, unit_boxes=True)   # decode clamps to [0,1]
    if return_all:
        return dict(rois=rois, count=count, keep=keep, topk=top, boxes=boxes, scores=scores, valid=valid)
    return rois, count


class ProposalPlan:
    """Pre-planned proposal layer for a fixed (B, N) shape: workspace and outputs are allocated once;
    ``run(cls, reg)`` is one ``frr_rpn_proposals`` call on the current stream (no allocation, no sync).

    Mixed-size batches: ``image_hw`` is then the padded (max) size of the batch and ``run(cls, reg, image_hw=sizes)``
    takes the per-image sizes as an int32 [B,2] device tensor, read by the kernels when they run: a graph captured with
    ``capture(cls, reg, sizes)`` serves every mix of sizes later written into ``sizes``."""

    def __init__(self, B: int, N: int, device, image_hw=None, anchors=None, mode: str = "train", stride: int = 16,
                 table=None, logits: bool = True, pre_nms_top_k=None, post_nms_top_k=None,
                 nms_thresh: float = RPN_NMS_THRESH, min_size: float = ops._MIN_SIZE, nms_cluster_size: int = 0):
        self.lib = _lib.load()
        self.nms_cluster_size = int(nms_cluster_size)  # 0: lowest latency of one call; 1: least SM time (ProposalPipeline)
        pre_k, post_k = PROPOSAL_MODES[mode]
        self.pre_k = pre_k if pre_nms_top_k is None else int(pre_nms_top_k)
        self.post_k = post_k if post_nms_top_k is None else int(post_nms_top_k)
        self.B, self.N, self.device = int(B), int(N), torch.device(device)
        self.logits, self.stride, self.thr, self.min_size = bool(logits), int(stride), float(nms_thresh), float(min_size)
        self._table, self._tptr, self.A = ops._table_arg(table)
        with torch.cuda.device(self.device):
            self.ws_bytes = int(self.lib.frr_rpn_proposals_workspace_bytes(self.B, self.N, self.pre_k, self.post_k))
            self._ws = torch.empty((self.ws_bytes + 256,), dtype=torch.uint8, device=self.device)
            self._ws_ptr = self._ws.data_ptr() + ((-self._ws.data_ptr()) % 256)
            self.rois = torch.empty((self.B, self.post_k, 4), dtype=torch.float32, device=self.device)
            self.count = torch.empty((self.B,), dtype=torch.int32, device=self.device)
        if anchors is not None:
            self.anchors = ops._req(anchors, "anchors", shape=(self.N, 4), device=self._ws.device)
            self.H = self.W = 0
        else:
            if image_hw is None:
                raise ValueError("image_hw is required when anchors are generated in-kernel")
            self.anchors = None
            self.H, self.W = int(image_hw[0]), int(image_hw[1])
        self.grid_hw = (self.H // self.stride, self.W // self.stride)   # padded grid of a mixed-size batch

    def run(self, cls, reg, rois=None, count=None, image_hw=None):
        """cls [B,N,2] logits / [B,N] scores and reg [B,N,4]: CUDA fp32 contiguous.  Returns (rois, count) --
        the plan's own output buffers unless ``rois`` / ``count`` are given (overwritten by the next run).
        ``image_hw``: per-image sizes (see the class doc); host sizes are checked and copied, so pass a device tensor
        where the call is captured into a graph."""
        B, N, dev = self.B, self.N, self._ws.device
        ops._check(cls, "cls", shape=(B, N, 2) if self.logits else (B, N), device=dev, contiguous=True)
        ops._check(reg, "reg", shape=(B, N, 4), device=dev, contiguous=True)
        rois = self.rois if rois is None else ops._check(rois, "rois", shape=(B, self.post_k, 4), device=dev, contiguous=True)
        count = self.count if count is None else ops._check(count, "count", torch.int32, (B,), dev, contiguous=True)
        hw = None
        if image_hw is not None:
            if self.anchors is not None:
                raise ValueError("ProposalPlan.run: per-image sizes need generated anchors (a plan built with image_hw)")
            hw = ops.sized_hw(image_hw, B, self.grid_hw, self.stride, dev)
        _lib.check(self.lib.frr_rpn_proposals(reg.data_ptr(), cls.data_ptr(), int(self.logits), ops._ptr(self.anchors),
                                              self._tptr, self.A, self.H, self.W, ops._ptr(hw), self.stride, self.min_size,
                                              self.B, self.N, self.pre_k, self.post_k, self.thr, rois.data_ptr(),
                                              count.data_ptr(), self._ws_ptr, self.ws_bytes, self.nms_cluster_size,
                                              torch.cuda.current_stream().cuda_stream), "frr_rpn_proposals")
        return rois, count


    def intermediates(self):
        """Views of the workspace regions the last ``run`` / graph replay left behind (no copies): decoded ``boxes``
        [B,N,4], ``scores`` [B,N], ``valid`` u8 [B,N], ``top_idx`` int32 [B,k] (indices into N, score descending),
        ``top_count`` int32 [B], ``keep`` int32 [B,post] (positions in the top-k order, -1 padded)."""
        import ctypes
        off = (ctypes.c_size_t * 6)()
        _lib.check(self.lib.frr_rpn_proposals_workspace_layout(self.B, self.N, self.pre_k, self.post_k, off),
                   "frr_rpn_proposals_workspace_layout")
        base = self._ws_ptr - self._ws.data_ptr()
        k = min(self.pre_k, self.N)
        B, N = self.B, self.N

        def view(o, nbytes, dtype, shape):
            return self._ws[base + o: base + o + nbytes].view(dtype).view(shape)

        return dict(boxes=view(off[0], B * N * 16, torch.float32, (B, N, 4)),
                    scores=view(off[1], B * N * 4, torch.float32, (B, N)),
                    valid=view(off[2], B * N, torch.uint8, (B, N)),
                    top_idx=view(off[3], B * k * 4, torch.int32, (B, k)),
                    top_count=view(off[4], B * 4, torch.int32, (B,)),
                    keep=view(off[5], B * self.post_k * 4, torch.int32, (B, self.post_k)))

    def capture(self, cls, reg, image_hw=None):
        """Capture one ``run(cls, reg)`` into a CUDA graph (the call neither allocates nor synchronises) and return the
        ``torch.cuda.CUDAGraph``; ``graph.replay()`` then re-runs the whole proposal layer on whatever ``cls`` / ``reg``
        (and the device tensor ``image_hw``) hold at that moment, writing ``self.rois`` / ``self.count``, for one graph
        launch instead of four kernel launches."""
        self.run(cls, reg, image_hw=image_hw)                 # warm-up outside the capture (function attributes, tables)
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        # thread_local: CUDA calls of other threads (e.g. NCCL's watchdog under torchrun) must not invalidate the capture
        with torch.cuda.graph(graph, capture_error_mode="thread_local"):
            self.run(cls, reg, image_hw=image_hw)
        return graph


class ProposalPipeline:
    """Throughput mode for DEVICE-resident head outputs: ``depth`` independent plans, each on its own stream, so
    that consecutive batches overlap on the GPU.  The top-k and NMS kernels run one CTA per image (NMS with
    ``nms_cluster_size=1``: 144 us per image-CTA instead of 108 us for a 2-CTA cluster, but 9.2 k instead of 13.8 k
    SM-microseconds per 64 images); the 84 SMs they leave idle at 64 images are filled by the neighbouring batches'
    kernels.  Measured at 64 images of 21 546 anchors (B200, 1965 MHz, 1000 W): 456 k images/s one batch at a time,
    772-777 k with 4 in flight.

    ``submit(cls, reg)`` orders the plan's stream after the caller's current stream (the producer of cls / reg),
    issues one ``frr_rpn_proposals`` call (or replays the graph captured for these tensors) and returns a ticket;
    ``result(ticket)`` orders the caller's current stream after that step and returns the plan's ``(rois, count)``
    (overwritten ``depth`` submits later).  No host synchronisation anywhere."""

    def __init__(self, B: int, N: int, device, depth: int = 3, **plan_kwargs):
        self.depth = int(depth)
        self.device = torch.device(device)
        plan_kwargs.setdefault("nms_cluster_size", 1)   # one CTA per image: the least SM time, other batches fill the SMs
        self.plans = [ProposalPlan(B, N, device, **plan_kwargs) for _ in range(self.depth)]
        with torch.cuda.device(self.device):
            self.streams = [torch.cuda.Stream(device=self.device) for _ in range(self.depth)]
        self._done = [torch.cuda.Event() for _ in range(self.depth)]
        self._graphs = {}
        self._captured_sizes = []
        self._n = 0

    def capture(self, cls, reg, image_hw=None):
        """Capture the call for these input tensors once per plan; ``submit`` on the same tensors then replays.
        ``image_hw``: per-image sizes of a mixed-size batch (see ``ProposalPlan``); the graphs read the device tensor at
        every replay, so pass the int32 [B,2] device tensor that ``submit`` will get (host sizes are copied to a device
        tensor the graphs keep, and are then fixed)."""
        image_hw = self._sizes(image_hw)
        if image_hw is not None:
            self._captured_sizes.append(image_hw)
        for j, plan in enumerate(self.plans):
            with torch.cuda.stream(self.streams[j]):
                self._graphs[(j, cls.data_ptr(), reg.data_ptr(), ops._ptr(image_hw))] = plan.capture(cls, reg, image_hw)
        torch.cuda.synchronize(self.device)

    def _sizes(self, image_hw):
        """per-image sizes as the device tensor the plans read (host sizes checked and copied on the current stream)"""
        if image_hw is None:
            return None
        p = self.plans[0]
        return ops.sized_hw(image_hw, p.B, p.grid_hw, p.stride, self.device)

    def submit(self, cls, reg, image_hw=None) -> int:
        image_hw = self._sizes(image_hw)
        t = self._n
        j = t % self.depth
        s = self.streams[j]
        s.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(s):
            g = self._graphs.get((j, cls.data_ptr(), reg.data_ptr(), ops._ptr(image_hw)))
            if g is not None:
                g.replay()
            else:
                self.plans[j].run(cls, reg, image_hw=image_hw)
            self._done[j].record(s)
        self._n += 1
        return t

    def result(self, ticket: int):
        if ticket < self._n - self.depth or ticket >= self._n:
            raise ValueError("ProposalPipeline.result: the step's buffers have been reused (or it was never submitted)")
        j = ticket % self.depth
        torch.cuda.current_stream(self.device).wait_event(self._done[j])
        return self.plans[j].rois, self.plans[j].count

    def drain(self):
        """Order the caller's current stream after every submitted step."""
        cur = torch.cuda.current_stream(self.device)
        for e in self._done[:min(self._n, self.depth)]:
            cur.wait_event(e)


class HostProposalPipeline:
    """Proposal layer for HOST inputs (numpy / CPU tensors), double buffered.

    ``submit(cls_host, reg_host)`` stages the inputs in pinned memory, copies them to the device on a copy
    stream, runs the plan on the compute stream and copies rois + counts back into pinned memory; it returns a
    ticket.  ``result(ticket)`` waits for that step only and returns ``(rois_host [B,post,4], count_host [B])``
    views (valid until the slot is reused two submits later).  With ``depth`` = 2 the H2D copy of step i+1
    overlaps the kernels of step i."""

    def __init__(self, plan: ProposalPlan, depth: int = 2):
        self.plan = plan
        dev = plan.device
        B, N = plan.B, plan.N
        cshape = (B, N, 2) if plan.logits else (B, N)
        self.depth = int(depth)
        with torch.cuda.device(dev):
            self.copy_stream = torch.cuda.Stream(device=dev)
            self.compute_stream = torch.cuda.Stream(device=dev)
            self.slots = []
            for _ in range(self.depth):
                self.slots.append(dict(
                    h_cls=torch.empty(cshape, dtype=torch.float32).pin_memory(),
                    h_reg=torch.empty((B, N, 4), dtype=torch.float32).pin_memory(),
                    d_cls=torch.empty(cshape, dtype=torch.float32, device=dev),
                    d_reg=torch.empty((B, N, 4), dtype=torch.float32, device=dev),
                    d_rois=torch.empty((B, plan.post_k, 4), dtype=torch.float32, device=dev),
                    d_count=torch.empty((B,), dtype=torch.int32, device=dev),
                    h_rois=torch.empty((B, plan.post_k, 4), dtype=torch.float32).pin_memory(),
                    h_count=torch.empty((B,), dtype=torch.int32).pin_memory(),
                    copied=torch.cuda.Event(), done=torch.cuda.Event(), busy=False))
        self._n = 0
        self.h2d_bytes = int(np.prod(cshape) * 4 + B * N * 16)
        self.d2h_bytes = int(B * plan.post_k * 16 + B * 4)

    def submit(self, cls_host, reg_host, stage: bool = True) -> int:
        """``stage=False``: cls_host / reg_host are already pinned CPU tensors and are copied from directly."""
        t = self._n
        s = self.slots[t % self.depth]
        if s["busy"]:
            s["done"].synchronize()      # slot reuse: its previous step must have left the device
        if stage:
            s["h_cls"].copy_(torch.as_tensor(cls_host))
            s["h_reg"].copy_(torch.as_tensor(reg_host))
            src_cls, src_reg = s["h_cls"], s["h_reg"]
        else:
            src_cls, src_reg = cls_host, reg_host
        with torch.cuda.stream(self.copy_stream):
            s["d_cls"].copy_(src_cls, non_blocking=True)
            s["d_reg"].copy_(src_reg, non_blocking=True)
            s["copied"].record(self.copy_stream)
        with torch.cuda.stream(self.compute_stream):
            self.compute_stream.wait_event(s["copied"])
            self.plan.run(s["d_cls"], s["d_reg"], rois=s["d_rois"], count=s["d_count"])
            s["h_rois"].copy_(s["d_rois"], non_blocking=True)
            s["h_count"].copy_(s["d_count"], non_blocking=True)
            s["done"].record(self.compute_stream)
        s["busy"] = True
        self._n += 1
        return t

    def result(self, ticket: int):
        s = self.slots[ticket % self.depth]
        s["done"].synchronize()
        return s["h_rois"], s["h_count"]


def _capture(fn, device):
    """Capture fn() into a CUDA graph; tensors fn allocates come from the graph's private pool and are the replay's
    outputs.  Returns (graph, outputs)."""
    fn()                                                      # warm-up outside the capture
    torch.cuda.synchronize(device)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, capture_error_mode="thread_local"):
        out = fn()
    return graph, out


class InferPlan:
    """FRCNN.predict's region path for a fixed batch shape (models/model.py:346-402), in the two halves the FC head
    (cuBLAS, not part of this library) sits between:

    ``pool(feat, cls, reg)``      proposal layer in test mode (6000 -> 300) -> feature-map rois with batch index
                                  (models/model.py:104-110) -> RoIPool 7x7: returns (pooled [B*R,C,7,7], rois [B,R,4], count [B])
    ``detect(head_cls, head_reg)``  per-class decode (:369-378) -> per-class NMS (:382-402) -> packed detections
                                  [B,max_det,6] (x1,y1,x2,y2,score,label) + counts, the evaluation hand-off

    Neither half synchronises with the host; ``capture_*`` record them into CUDA graphs (one graph launch per half).

    Mixed-size batches: build the plan with the padded (max) ``image_hw`` and pass the per-image sizes to ``pool`` /
    ``capture_pool`` as an int32 [B,2] device tensor: anchors, the roi scaling and the RoIPool window clip then use each
    image's own size, and a captured graph reads the sizes at every replay.

    ``rank`` / ``per_class_max`` choose which ``max_det`` detections of an image ``detect`` packs (see
    ``ops.pack_detections``): ``"class"`` (default) the first in class order, ``"score"`` the highest-scoring, at most
    ``per_class_max`` per class when that is > 0.  ``class_nms`` runs at its full capacity, so the ranking sees every
    detection; the ranking's workspace is allocated here, once."""

    def __init__(self, B: int, image_hw, num_classes: int, device, stride: int = 16, max_det: int = 100,
                 score_thres: float = 0.05, iou_thr: float = 0.3, mode: str = "test", logits: bool = True,
                 nms_cluster_size: int = 0, rank: str = "class", per_class_max: int = 0):
        from . import dist as fdist
        self._fdist = fdist
        self.B, self.hw, self.NC, self.device = int(B), (int(image_hw[0]), int(image_hw[1])), int(num_classes), torch.device(device)
        self.stride = int(stride)
        self.fhw = (self.hw[0] // stride, self.hw[1] // stride)
        self.N = self.fhw[0] * self.fhw[1] * 9
        self.proposal = ProposalPlan(self.B, self.N, self.device, image_hw=self.hw, mode=mode, stride=stride, logits=logits,
                                     nms_cluster_size=nms_cluster_size)
        self.R = self.proposal.post_k
        self.max_det, self.score_thres, self.iou_thr = int(max_det), float(score_thres), float(iou_thr)
        ops.check_rank(rank, per_class_max)
        self.rank, self.per_class_max = rank, int(per_class_max)
        with torch.cuda.device(self.device):
            self.rois5 = torch.empty((self.B * self.R, 5), dtype=torch.float32, device=self.device)
            self.rank_ws = (ops.pack_ranked_workspace(self.B, self.R * (self.NC - 1), self.max_det, self.device)
                            if rank == "score" else None)

    def pool(self, feat, cls, reg, want_argmax: bool = False, image_hw=None):
        rois, cnt = self.proposal.run(cls, reg, image_hw=image_hw)
        ops.rois5(rois, cnt, self.fhw, out=self.rois5, image_hw=image_hw, stride=self.stride)
        pooled, arg = ops.roi_pool_forward(feat, self.rois5, want_argmax=want_argmax, image_hw=image_hw, stride=self.stride)
        return (pooled, rois, cnt, arg) if want_argmax else (pooled, rois, cnt)

    def detect(self, head_cls, head_reg, return_all: bool = False):
        B, R, NC = self.B, self.R, self.NC
        rois, cnt = self.proposal.rois, self.proposal.count
        prob, boxes = ops.decode_classwise(head_cls, head_reg, rois.reshape(-1, 4), NC)
        db, dl, ds, dc = ops.class_nms(prob.reshape(B, R, NC), boxes.reshape(B, R, 4 * NC), NC, score_thres=self.score_thres,
                                       iou_thr=self.iou_thr, roi_count=cnt)
        packed, pc = self._fdist.pack_detections(db, dl, ds, dc, self.max_det, rank=self.rank,
                                                 per_class_max=self.per_class_max, workspace=self.rank_ws)
        if return_all:
            return dict(packed=packed, count=pc, prob=prob, boxes=boxes, det=(db, dl, ds, dc))
        return packed, pc

    def capture_pool(self, feat, cls, reg, image_hw=None):
        return _capture(lambda: self.pool(feat, cls, reg, image_hw=image_hw), self.device)

    def capture_detect(self, head_cls, head_reg):
        return _capture(lambda: self.detect(head_cls, head_reg), self.device)


class TrainPlan:
    """The training-side region stage for a fixed batch shape (models/model.py:310-335): both target makers with the
    reference's sampling replayed on the device (no host synchronisation), RoIPool forward of the sampled rois and its
    backward.  ``targets_and_pool`` / ``pool_backward`` can be recorded into CUDA graphs with ``capture_*``.
    ``pool_backward`` follows ``torch.use_deterministic_algorithms`` when it runs; a captured graph keeps the backward
    kernel chosen at capture time, whatever the flag is when the graph is replayed.

    Mixed-size batches: build the plan with the padded (max) ``image_hw`` and pass the per-image sizes to
    ``targets_and_pool`` / ``capture_targets_and_pool`` as an int32 [B,2] device tensor (read at every replay);
    ``pool_backward`` uses the sizes of the last ``targets_and_pool``."""

    def __init__(self, B: int, image_hw, device, generator=None, stride: int = 16):
        from . import targets
        self._targets = targets
        self.B, self.hw, self.device = int(B), (int(image_hw[0]), int(image_hw[1])), torch.device(device)
        self.stride = int(stride)
        self.fhw = (self.hw[0] // stride, self.hw[1] // stride)
        self.generator = generator if generator is not None else targets.DeviceGenerator(self.device)
        with torch.cuda.device(self.device):
            self.rois5 = torch.empty((self.B * targets.FRCNN_BATCH, 5), dtype=torch.float32, device=self.device)
        self.last = None

    def targets_and_pool(self, feat, gt, gt_label, proposals, proposal_count, gt_count=None, image_hw=None):
        if image_hw is not None:
            image_hw = ops.sized_hw(image_hw, self.B, self.fhw, self.stride, self.device)
        t = self._targets.make_targets(gt, gt_count, gt_label, proposals, proposal_count,
                                       image_hw=self.hw if image_hw is None else image_hw, generator=self.generator,
                                       grid_hw=self.fhw)
        ops.rois5(t["sample_rois"], t["n_samples"], self.fhw, out=self.rois5, image_hw=image_hw, stride=self.stride)
        pooled, arg = ops.roi_pool_forward(feat, self.rois5, image_hw=image_hw, stride=self.stride)
        self.last = dict(targets=t, pooled=pooled, argmax=arg, feat_shape=tuple(feat.shape),
                         channels_last=(not feat.is_contiguous()), image_hw=image_hw)
        return t, pooled

    def pool_backward(self, grad_out):
        s = self.last
        return ops.roi_pool_backward(grad_out, s["argmax"], self.rois5, s["feat_shape"], channels_last=s["channels_last"],
                                     image_hw=s["image_hw"], stride=self.stride)

    def capture_targets_and_pool(self, feat, gt, gt_label, proposals, proposal_count, image_hw=None):
        return _capture(lambda: self.targets_and_pool(feat, gt, gt_label, proposals, proposal_count, image_hw=image_hw),
                        self.device)

    def capture_pool_backward(self, grad_out):
        return _capture(lambda: self.pool_backward(grad_out), self.device)
