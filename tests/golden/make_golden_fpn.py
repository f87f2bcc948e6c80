"""Golden fixtures for the FPN-variant target makers (run in the BUILD container only).

    python tests/golden/make_golden_fpn.py

Imports the UNMODIFIED ``RPNTargetMaker`` / ``FRCNNTargetMaker`` of /root/reference/models/new_model.py (the
variant main.py trains today, SURVEY.md section 8f rank 2) and stores their outputs on seeded synthetic inputs in
tests/golden/targets_fpn.npz.  Same harness-side patches as make_golden.py.
"""
from __future__ import annotations

import contextlib
import io
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
from faster_rcnn_pytorch_b200 import synth  # noqa: E402


def main():
    torch.Tensor.get_device = lambda self: self.device
    sys.modules.setdefault("gdown", types.ModuleType("gdown"))
    sys.path.insert(0, "/root/reference")
    import models.new_model as nm
    import anchor as ref_anchor

    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    am = ref_anchor.FRCNNAnchorMaker()
    rtm, ftm = nm.RPNTargetMaker(), nm.FRCNNTargetMaker()
    g = {}
    for name, hw, gseed, G, tseed in [("a", (320, 480), 7000, 5, 7000), ("b", (600, 1000), 7001, 8, 7001),
                                      ("many", (320, 480), 7002, 150, 7002), ("one", (160, 256), 7003, 1, 7003)]:
        anchors = am._enumerate_shifted_anchor(hw)      # any [N,4] anchor set: the maker does not care where it came from
        gt, lab = synth.gt_boxes(gseed, G)
        lab = lab + 1                                    # FPN variant: labels are used as they are (background = 0)
        torch.manual_seed(tseed)
        with contextlib.redirect_stdout(io.StringIO()):
            cls_t, reg_t = rtm(t(gt), t(anchors))
        g[f"{name}_rpn_cls"] = cls_t.numpy().astype(np.int8)
        nz = np.nonzero(cls_t.numpy() >= 0)[0]
        g[f"{name}_rpn_reg_sampled"] = reg_t.numpy()[nz].copy()
        rois_np, _ = synth.random_boxes(tseed + 50, 2000)
        torch.manual_seed(tseed + 1)
        with contextlib.redirect_stdout(io.StringIO()):
            fc, fr, fs = ftm(t(gt), t(lab), t(rois_np))
        g[f"{name}_frcnn_cls"] = fc.numpy().astype(np.int16)
        g[f"{name}_frcnn_reg"] = fr.numpy().copy()
        g[f"{name}_frcnn_rois"] = fs.numpy().copy()
    # a GT that overlaps nothing: the tie-inclusive rule then marks EVERY anchor with IoU == 0 positive (:316-318)
    hw = (160, 256)
    anchors = am._enumerate_shifted_anchor(hw)
    inside = (anchors[:, 0] >= 0) & (anchors[:, 1] >= 0) & (anchors[:, 2] <= 1) & (anchors[:, 3] <= 1)
    anchors_in = anchors[inside]
    gt = np.array([[0.2, 0.2, 0.6, 0.7], [5.0, 5.0, 5.1, 5.1]], np.float32)
    torch.manual_seed(9)
    with contextlib.redirect_stdout(io.StringIO()):
        cls_t, reg_t = rtm(t(gt), t(anchors_in))
    g["far_rpn_cls"] = cls_t.numpy().astype(np.int8)
    g["far_anchors"] = anchors_in.copy()
    np.savez_compressed(os.path.join(HERE, "targets_fpn.npz"), **g)
    print("targets_fpn.npz", os.path.getsize(os.path.join(HERE, "targets_fpn.npz")))




def proposals():
    """RegionProposalNetwork.forward of models/new_model.py on a small synthetic pyramid: stores the head outputs,
    the torchvision anchors and the reference's rois (tests/golden/proposal_fpn.npz)."""
    torch.Tensor.get_device = lambda self: self.device
    sys.modules.setdefault("gdown", types.ModuleType("gdown"))
    sys.path.insert(0, "/root/reference")
    import models.new_model as nm
    g = {}
    for name, hw, seed, mode in [("train", (128, 192), 8000, "train"), ("test", (160, 160), 8001, "test")]:
        torch.manual_seed(seed)
        rpn = nm.RegionProposalNetwork().eval()
        with torch.no_grad():
            for m in (rpn.rpn_head.cls_layer, rpn.rpn_head.reg_layer):
                m.weight.normal_(0, 0.5)       # spread the scores / deltas (the default 0.01 init gives thousands of ties)
        x = torch.zeros(1, 3, hw[0], hw[1])
        feats = {str(l): torch.randn(1, 256, -(-hw[0] // s), -(-hw[1] // s)) for l, s in enumerate((4, 8, 16, 32, 64))}
        with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
            cls, reg, rois, anchor = rpn(x, feats, mode)
        g[f"{name}_cls"] = cls.numpy().copy()
        rg = (reg.numpy() * 0.05).astype(np.float32)                   # keep exp() of the deltas tame
        rg[::97, 2] = -6.0                                              # a few boxes thinner than min_size 10/1000
        g[f"{name}_reg"] = rg
        g[f"{name}_anchor"] = anchor.numpy().copy()
        # the reference's own proposal arithmetic (models/new_model.py:46-83) on the stored (scaled) deltas and on
        # tie-free scores (the reference's sort order of equal scores is unspecified, SURVEY section 8c)
        import utils.util as U
        import torchvision
        sc = torch.softmax(cls, dim=-1)[..., 1].numpy().copy()
        for _ in range(64):
            _, first = np.unique(sc, return_index=True)
            dup = np.ones(len(sc), bool); dup[first] = False
            if not dup.any():
                break
            sc[dup] = np.nextafter(sc[dup], np.float32(2.0))
        assert len(np.unique(sc)) == len(sc)
        sc = torch.from_numpy(sc)
        roi = U.cxcy_to_xy(U.decode(torch.from_numpy(g[f"{name}_reg"]), U.xy_to_cxcy(anchor))).clamp(0, 1)
        ws, hs = roi[:, 2] - roi[:, 0], roi[:, 3] - roi[:, 1]
        keep = (hs >= (10 / 1000)) & (ws >= (10 / 1000))
        roi_c, sc_c = roi[keep], sc[keep]
        ss, si = sc_c.sort(descending=True)
        pre_k, post_k = (4000, 1000) if mode == "train" else (2000, 1000)
        k = min(pre_k, si.numel())
        kp = torchvision.ops.nms(roi_c[si[:k]], ss[:k], 0.7)[:post_k]
        g[f"{name}_score"] = sc.numpy().copy()
        g[f"{name}_boxes"] = roi.numpy().copy()              # the reference's decoded + clamped boxes
        g[f"{name}_valid"] = keep.numpy().copy()
        g[f"{name}_topk_idx"] = si[:k].numpy().astype(np.int32)
        g[f"{name}_keep"] = kp.numpy().astype(np.int32)
        g[f"{name}_rois"] = roi_c[si[:k]][kp].numpy().copy()
    np.savez_compressed(os.path.join(HERE, "proposal_fpn.npz"), **g)
    print("proposal_fpn.npz", os.path.getsize(os.path.join(HERE, "proposal_fpn.npz")))


def multiscale():
    """torchvision.ops.MultiScaleRoIAlign (CPU) as called at models/new_model.py:127,143 -> tests/golden/msroialign.npz"""
    import torchvision
    from torchvision.ops.poolers import LevelMapper
    image_hw = (256, 320)
    feats, rois5 = synth.pyramid_inputs(image_hw=image_hw)
    pool = torchvision.ops.MultiScaleRoIAlign(featmap_names=["0", "1", "2", "3"], output_size=7, sampling_ratio=2)
    x = {str(i): torch.from_numpy(f) for i, f in enumerate(feats)}
    boxes = [torch.from_numpy(rois5[rois5[:, 0] == b, 1:]) for b in range(feats[0].shape[0])]
    order = np.concatenate([np.nonzero(rois5[:, 0] == b)[0] for b in range(feats[0].shape[0])])
    g = {}
    for tag, shapes in [("hw", [image_hw] * 2), ("wh_like_reference", [(image_hw[1], image_hw[0])] * 2)]:
        for f in x.values():
            f.requires_grad_(True); f.grad = None
        out = pool(x, boxes, shapes)
        go = torch.from_numpy(np.random.RandomState(8101).standard_normal(tuple(out.shape)).astype(np.float32))
        out.backward(go)
        full = np.zeros(out.shape, np.float32); full[order] = out.detach().numpy()
        gfull = np.zeros(out.shape, np.float32); gfull[order] = go.numpy()
        g[f"{tag}_out"] = full                          # rows in the order of rois5
        g["grad_out"] = gfull                           # the same seeded gradient for both tags: stored once
        for i, f in enumerate(x.values()):
            g[f"{tag}_gin{i}"] = f.grad.numpy().copy()
        scales = pool.scales
        k_min, k_max = int(-np.log2(scales[0])), int(-np.log2(scales[-1]))
        lv = LevelMapper(k_min, k_max)([torch.from_numpy(rois5[:, 1:])]).numpy()
        g[f"{tag}_levels"] = lv.astype(np.int32)
        g[f"{tag}_scales"] = np.asarray(scales, np.float64)
        pool.scales = None; pool.map_levels = None
    np.savez_compressed(os.path.join(HERE, "msroialign.npz"), **g)
    print("msroialign.npz", os.path.getsize(os.path.join(HERE, "msroialign.npz")))


if __name__ == "__main__":
    main()
    proposals()
    multiscale()
