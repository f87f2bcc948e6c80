"""GPU: every tensor the Python wrappers hand to libfrr is checked against the shape, dtype and device include/frr.h
states, before anything is launched.

No kernel of the library runs here: ``_lib.load`` returns a recorder that answers the host-only queries (workspace sizes,
layouts, variant choices, host tables, errors) from the real library and records every other entry point, returning 0.
Each case makes one well-formed call and expects exactly its entry points; then it changes one thing at a time (one
dimension of one tensor, its dtype, its device, or strides on a tensor written in place) and expects ValueError before
the entry point that would have read or written the tensor is reached.  A strided input is copied and accepted."""
import re
from dataclasses import dataclass, field

import pytest
import torch

from faster_rcnn_pytorch_b200 import _lib, ops, region, targets

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F32, F64, I32, I64, U8, I8 = torch.float32, torch.float64, torch.int32, torch.int64, torch.uint8, torch.int8
HOST_ONLY = re.compile(r"frr_(\w+_workspace_bytes|\w+_layout|\w+_variant|\w+_host|last_error|abi_version)")

B, N, G, R, K, C, S = 2, 18, 3, 5, 6, 4, 8      # N = 9 anchors on a 1 x 2 grid (a 16 x 32 image at stride 16)
HW, GRID = (16, 32), (1, 2)


class Recorder:
    def __init__(self, lib):
        self.lib, self.calls = lib, []

    def __getattr__(self, name):
        if HOST_ONLY.fullmatch(name):
            return getattr(self.lib, name)

        def record(*args):
            self.calls.append(name)
            return 0
        record.__name__ = name
        return record


@pytest.fixture
def rec(monkeypatch):
    r = Recorder(_lib.load())
    monkeypatch.setattr(_lib, "load", lambda: r)
    return r


@dataclass
class Case:
    call: object                        # fn(tensors by name)
    args: dict                          # name -> (shape, dtype)
    calls: tuple                        # the entry points a well-formed call reaches, in order
    free: set = field(default_factory=set)         # (name, dim) whose size no other argument fixes
    inplace: set = field(default_factory=set)      # written in place (or read by a plan without a copy): no copy allowed
    # name, or (name, dim) -> index in ``calls`` of the first entry point that takes both tensors a change makes disagree
    # (0 unless given: the wrapper checks every tensor before its first entry point)
    first_use: dict = field(default_factory=dict)


def _ws_rpn(t, anchored):
    return dict(gt=t["gt"], anchors=t["anchors"] if anchored else None, image_hw=None if anchored else t["image_hw"],
                geom=(0, 0, 16, None, N) if anchored else (GRID[0] * 16, GRID[1] * 16, 16, None, N),
                argmax=t["argmax"], label8=t["label8"], pos_list=t["pos_list"], neg_list=t["neg_list"])


def _plan_run(t):
    plan = region.ProposalPlan(B, N, DEV, image_hw=HW, mode="test")
    return plan.run(t["cls"], t["reg"], rois=t["rois"], count=t["count"], image_hw=t["image_hw"])


RPN_FINALIZE_ARGS = dict(gt=((B, G, 4), F32), argmax=((B, N), I32), label8=((B, N), I8), pos_list=((B, N), I32),
                         neg_list=((B, N), I32), disable=((7,), I32), disable_off=((3 * B,), I32))
LOSS = ("rpn_cls", "rpn_reg", "rpn_target_cls", "rpn_target_reg", "frcnn_cls", "frcnn_reg", "frcnn_target_cls",
        "frcnn_target_reg")
DETS = dict(det_boxes=((B, 7, 4), F32), det_labels=((B, 7), I32), det_scores=((B, 7), F32), det_count=((B,), I32),
            image_wh=((B, 2), F32))

CASES = {
    "rpn_decode": Case(
        lambda t: ops.rpn_decode(t["reg"], t["cls"], anchors=t["anchors"]),
        dict(reg=((B, N, 4), F32), cls=((B, N, 2), F32), anchors=((N, 4), F32)), ("frr_rpn_decode",)),
    "rpn_decode_sized": Case(
        lambda t: ops.rpn_decode(t["reg"], t["cls"], image_hw=t["image_hw"], grid_hw=GRID),
        dict(reg=((B, N, 4), F32), cls=((B, N), F32), image_hw=((B, 2), I32)), ("frr_rpn_decode_sized",)),
    "topk_desc": Case(
        lambda t: ops.topk_desc(t["scores"], 4, valid=t["valid"], boxes=t["boxes"]),
        dict(scores=((B, N), F32), valid=((B, N), U8), boxes=((B, N, 4), F32)), ("frr_topk_desc_opt",)),
    "nms_sorted": Case(
        lambda t: ops.nms_sorted(t["boxes"], 0.7, counts=t["counts"]),
        dict(boxes=((B, N, 4), F32), counts=((B,), I32)), ("frr_nms_sorted",), free={("boxes", 1)}),
    "rois5": Case(
        lambda t: ops.rois5(t["rois"], t["count"], GRID, out=t["out"], image_hw=t["image_hw"]),
        dict(rois=((B, R, 4), F32), count=((B,), I32), out=((B * R, 5), F32), image_hw=((B, 2), I32)), ("frr_rois5",),
        inplace={"out"}),
    "roi_pool_forward": Case(
        lambda t: ops.roi_pool_forward(t["feat"], t["rois5"], image_hw=t["image_hw"]),
        dict(feat=((B, C, 3, 5), F32), rois5=((K, 5), F32), image_hw=((B, 2), I32)), ("frr_roi_pool_fwd",),
        free={("feat", 1), ("feat", 2), ("feat", 3), ("rois5", 0)}),
    "roi_pool_backward": Case(
        lambda t: ops.roi_pool_backward(t["grad_out"], t["argmax"], t["rois5"], (B, C, 3, 5), deterministic=False),
        dict(grad_out=((K, C, 7, 7), F32), argmax=((K, C, 7, 7), I32), rois5=((K, 5), F32)), ("frr_roi_pool_bwd",)),
    "roi_pool_backward_deterministic": Case(
        lambda t: ops.roi_pool_backward(t["grad_out"], t["argmax"], t["rois5"], (B, C, 3, 5), deterministic=True,
                                        image_hw=t["image_hw"]),
        dict(grad_out=((K, C, 7, 7), F32), argmax=((K, C, 7, 7), I32), rois5=((K, 5), F32), image_hw=((B, 2), I32)),
        ("frr_roi_pool_bwd_deterministic",)),
    "roi_align_forward": Case(
        lambda t: ops.roi_align_forward(t["feat"], t["rois5"], out=t["out"]),
        dict(feat=((B, C, 3, 5), F32), rois5=((K, 5), F32), out=((K, C, 7, 7), F32)), ("frr_roi_align_fwd",),
        free={("feat", 0), ("feat", 2), ("feat", 3)}, inplace={"out"}),
    "roi_align_backward": Case(
        lambda t: ops.roi_align_backward(t["grad_out"], t["rois5"], (B, C, 3, 5), deterministic=False),
        dict(grad_out=((K, C, 7, 7), F32), rois5=((K, 5), F32)), ("frr_roi_align_bwd",),
        free={("grad_out", 2), ("grad_out", 3)}),
    "rpn_targets_assign": Case(
        lambda t: ops.rpn_targets_assign(t["gt"], t["gt_count"], N, anchors=t["anchors"]),
        dict(gt=((B, G, 4), F32), gt_count=((B,), I32), anchors=((N, 4), F32)), ("frr_rpn_targets_assign",),
        free={("gt", 1)}),
    "rpn_targets_finalize": Case(
        lambda t: ops.rpn_targets_finalize(_ws_rpn(t, False), t["disable"], t["disable_off"]),
        dict(RPN_FINALIZE_ARGS, image_hw=((B, 2), I32)), ("frr_rpn_targets_finalize",),
        free={("gt", 1), ("disable", 0)}, inplace={"label8"}),
    "rpn_targets_finalize_anchored": Case(
        lambda t: ops.rpn_targets_finalize(_ws_rpn(t, True), t["disable"], t["disable_off"]),
        dict(RPN_FINALIZE_ARGS, anchors=((N, 4), F32)), ("frr_rpn_targets_finalize",),
        free={("gt", 1), ("disable", 0)}, inplace={"label8"}),
    "frcnn_targets_assign": Case(
        lambda t: ops.frcnn_targets_assign(t["rois"], t["roi_count"], t["gt"], t["gt_count"]),
        dict(rois=((B, R, 4), F32), roi_count=((B,), I32), gt=((B, G, 4), F32), gt_count=((B,), I32)),
        ("frr_frcnn_targets_assign",), free={("rois", 1), ("gt", 1)}),
    "frcnn_targets_finalize": Case(
        lambda t: ops.frcnn_targets_finalize(
            dict(rois=t["rois"], roi_count=t["roi_count"], gt=t["gt"], argmax=t["argmax"], pos_list=t["pos_list"],
                 neg_list=t["neg_list"]), t["gt_label"], t["sel"], t["sel_n"]),
        dict(rois=((B, R, 4), F32), roi_count=((B,), I32), gt=((B, G, 4), F32), argmax=((B, R + G), I32),
             pos_list=((B, R + G), I32), neg_list=((B, R + G), I32), gt_label=((B, G), I64), sel=((B, S), I32),
             sel_n=((B, 2), I32)), ("frr_frcnn_targets_finalize",), free={("sel", 1)}),
    "sample_targets": Case(
        lambda t: ops.sample_targets(t["mt_state"], ws_rpn=dict(counts=t["rpn_counts"], label8=t["label8"],
                                                                pos_list=t["pos_list"], neg_list=t["neg_list"]),
                                     ws_frcnn=dict(counts=t["frcnn_counts"])),
        dict(mt_state=((626,), I32), rpn_counts=((B, 2), I32), label8=((B, N), I8), pos_list=((B, N), I32),
             neg_list=((B, N), I32), frcnn_counts=((B, 2), I32)), ("frr_sample_targets",),
        inplace={"mt_state", "label8"}),
    "region_loss": Case(
        lambda t: ops.region_loss(*(t[k] for k in LOSS)),
        dict(rpn_cls=((B, N, 2), F32), rpn_reg=((B, N, 4), F32), rpn_target_cls=((B, N), I64),
             rpn_target_reg=((B, N, 4), F32), frcnn_cls=((B, S, C), F32), frcnn_reg=((B, S, C, 4), F32),
             frcnn_target_cls=((B, S), I64), frcnn_target_reg=((B, S, 4), F32)), ("frr_region_loss",)),
    "decode_classwise": Case(
        lambda t: ops.decode_classwise(t["cls_logits"], t["reg"], t["rois"], C),
        dict(cls_logits=((K, C), F32), reg=((K, 4 * C), F32), rois=((K, 4), F32)), ("frr_decode_classwise",)),
    "class_nms": Case(
        lambda t: ops.class_nms(t["prob"], t["boxes"], C, roi_count=t["roi_count"]),
        dict(prob=((B, R, C), F32), boxes=((B, R, 4 * C), F32), roi_count=((B,), I32)), ("frr_class_nms",)),
    "pack_detections": Case(
        lambda t: ops.pack_detections(*(t[k] for k in DETS if k != "image_wh"), 5, image_wh=t["image_wh"]),
        DETS, ("frr_pack_detections",)),
    "pack_detections_ranked": Case(
        lambda t: ops.pack_detections(*(t[k] for k in DETS if k != "image_wh"), 5, image_wh=t["image_wh"],
                                      rank="score", workspace=t["workspace"]),
        dict(DETS, workspace=((1 << 16,), U8)), ("frr_pack_detections_ranked",), free={("workspace", 0)}),
    "fpn_level_rois": Case(
        lambda t: ops.fpn_level_rois(t["rois5"], 2, 3), dict(rois5=((K, 5), F32)), ("frr_fpn_level_rois",),
        free={("rois5", 0)}),
    "multiscale_roi_align_forward": Case(
        lambda t: ops.multiscale_roi_align_forward([t["features0"], t["features1"]], t["rois5"], (7, 7), 2,
                                                   [0.25, 0.125], 2, 3),
        dict(features0=((B, C, 8, 8), F32), features1=((B, C, 4, 4), F32), rois5=((K, 5), F32)),
        ("frr_fpn_level_rois", "frr_roi_align_fwd", "frr_roi_align_fwd"),
        free={("features0", 0), ("features0", 2), ("features0", 3), ("features1", 0), ("features1", 2),
              ("features1", 3), ("rois5", 0)}),
    "ProposalPlan.run": Case(
        _plan_run,
        dict(cls=((B, N, 2), F32), reg=((B, N, 4), F32), rois=((B, 300, 4), F32), count=((B,), I32),
             image_hw=((B, 2), I32)), ("frr_rpn_proposals",), inplace={"cls", "reg", "rois", "count"}),
    "make_targets": Case(
        lambda t: targets.make_targets(t["gt"], t["gt_count"], t["gt_label"], t["rois"], t["roi_count"], image_hw=HW,
                                       generator=targets.DeviceGenerator(DEV)),
        dict(gt=((B, G, 4), F32), gt_count=((B,), I32), gt_label=((B, G), I64), rois=((B, R, 4), F32),
             roi_count=((B,), I32)),
        ("frr_rpn_targets_assign", "frr_frcnn_targets_assign", "frr_sample_targets", "frr_rpn_targets_finalize",
         "frr_frcnn_targets_finalize"), free={("rois", 1)},
        first_use={"rois": 1, "roi_count": 1, "gt_label": 4, ("gt", 1): 4}),
}


def _variants():
    for case, c in CASES.items():
        yield pytest.param(case, None, "ok", id=f"{case}-ok")
        for name, (shape, _) in c.args.items():
            for d in range(len(shape)):
                if (name, d) not in c.free:
                    yield pytest.param(case, name, d, id=f"{case}-{name}-dim{d}")
            for change in ("dtype", "strided") + (("cuda1",) if len(c.args) > 1 else ()):
                yield pytest.param(case, name, change, id=f"{case}-{name}-{change}")


def _tensor(shape, dtype, change=None):
    if change == "dtype":
        dtype = F64 if dtype == F32 else F32
    if isinstance(change, int):
        shape = tuple(s + (i == change) for i, s in enumerate(shape))
    if change == "strided":                     # same shape and dtype, every stride doubled
        return torch.empty(tuple(shape) + (2,), dtype=dtype, device=DEV)[..., 0]
    return torch.empty(shape, dtype=dtype, device="cuda:1" if change == "cuda1" else DEV)


@pytest.mark.parametrize("case,name,change", list(_variants()))
def test_wrapper_checks_every_tensor_before_the_launch(rec, case, name, change):
    c = CASES[case]
    if change == "cuda1" and torch.cuda.device_count() < 2:
        pytest.skip("needs a second CUDA device")
    t = {n: _tensor(shape, dtype, change if n == name else None) for n, (shape, dtype) in c.args.items()}
    if change == "ok" or (change == "strided" and name not in c.inplace):    # a strided input is copied, not refused
        c.call(t)
        assert rec.calls == list(c.calls)
        return
    with pytest.raises(ValueError):
        c.call(t)
    assert rec.calls == list(c.calls[:c.first_use.get((name, change), c.first_use.get(name, 0))])


def test_multiscale_roi_align_needs_one_map_per_level(rec):
    feats = [torch.empty((B, C, 8 >> l, 8 >> l), device=DEV) for l in range(2)]
    rois5 = torch.empty((K, 5), device=DEV)
    for k_max in (2, 4):
        with pytest.raises(ValueError, match="one feature map per level"):
            ops.multiscale_roi_align_forward(feats, rois5, (7, 7), 2, [0.25, 0.125, 0.0625], 2, k_max)
    assert rec.calls == []
