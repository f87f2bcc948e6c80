"""Developer tool: one launch of each RoI kernel at the config-3 shape (for ncu)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from faster_rcnn_pytorch_b200 import ops, synth
dev = torch.device("cuda:0")
B, C, fh, fw, per_img = 16, 512, 37, 62, 128
K = B * per_img
feat = torch.from_numpy(synth.features(1, B, C, fh, fw)).to(dev)
rois = torch.from_numpy(np.concatenate([np.concatenate([np.full((per_img, 1), b, np.float32),
        synth.random_boxes(10 + b, per_img)[0] * np.array([fw, fh, fw, fh], np.float32)], 1) for b in range(B)])).to(dev)
go = torch.randn((K, C, 7, 7), device=dev)
# one launch each of the sampling and loss kernels (config-3 shapes) so that the ncu capture of this script has them
from faster_rcnn_pytorch_b200 import targets
hw, G = (600, 1000), 8
gt = torch.from_numpy(np.stack([synth.gt_boxes(3000 + i, G)[0] for i in range(B)])).to(dev)
lab = torch.from_numpy(np.stack([synth.gt_boxes(3000 + i, G)[1] for i in range(B)])).to(dev)
props = torch.from_numpy(np.stack([synth.random_boxes(3100 + i, 2000)[0] for i in range(B)])).to(dev)
torch.manual_seed(0)
gen = targets.DeviceGenerator(dev)
t = targets.make_targets(gt, None, lab, props, None, image_hw=hw, generator=gen)
N = t["rpn_cls"].shape[1]
loss = ops.region_loss(torch.randn((B, N, 2), device=dev), torch.randn((B, N, 4), device=dev), t["rpn_cls"], t["rpn_reg"],
                       torch.randn((B, 128, 21), device=dev), torch.randn((B, 128, 21, 4), device=dev),
                       t["frcnn_cls"].clamp(min=0), t["frcnn_reg"])
for _ in range(2):
    out, arg = ops.roi_pool_forward(feat, rois)
    gin = ops.roi_pool_backward(go, arg, rois, feat.shape)
    oa = ops.roi_align_forward(feat, rois, sampling_ratio=2)
    ga = ops.roi_align_backward(go, rois, feat.shape, sampling_ratio=2)
torch.cuda.synchronize()
print("ok")
