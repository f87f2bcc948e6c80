"""Developer tool: times roi_pool_forward (with / without argmax) at the config-3 shape on RPN-sized and small rois."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from faster_rcnn_pytorch_b200 import ops, synth, region
dev = torch.device("cuda:0")
B, C, fh, fw, per = 16, 512, 37, 62, 128
hw = (600, 1000)
rs = np.random.RandomState(1)
feats = [torch.from_numpy(rs.standard_normal((B, C, fh, fw)).astype(np.float32)).to(dev) for _ in range(3)]
n = synth.num_anchors(hw)
lg = torch.from_numpy(rs.standard_normal((B, n, 2)).astype(np.float32)).to(dev)
rg = torch.from_numpy((rs.standard_normal((B, n, 4)) * 0.2).astype(np.float32)).to(dev)
props, pcnt = region.rpn_proposals(lg, rg, image_hw=hw, mode="train")
scale = torch.tensor([fw, fh, fw, fh], dtype=torch.float32, device=dev)
bidx = torch.arange(B, device=dev, dtype=torch.float32).repeat_interleave(per)[:, None]
rois5 = torch.cat([bidx, (props[:, :per] * scale).reshape(-1, 4)], dim=1).contiguous()
small = torch.from_numpy(np.concatenate([np.concatenate([np.full((per, 1), b, np.float32),
        synth.random_boxes(10 + b, per)[0] * np.array([fw, fh, fw, fh], np.float32)], 1) for b in range(B)])).to(dev)
def t(fn, reps=20):
    for i in range(3): fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps): fn(i)
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3
out0 = ops.roi_pool_forward(feats[0], rois5)
print(
      "rpn-rois us", round(t(lambda i: ops.roi_pool_forward(feats[i % 3], rois5)), 1),
      "small-rois us", round(t(lambda i: ops.roi_pool_forward(feats[i % 3], small)), 1),
      "noarg us", round(t(lambda i: ops.roi_pool_forward(feats[i % 3], rois5, want_argmax=False)), 1),
      "checksum", float(out0[0].double().sum()), int(out0[1].long().sum()))
wh = (rois5[:, 3] - rois5[:, 1]), (rois5[:, 4] - rois5[:, 2])
print("rpn roi w/h mean", float(wh[0].mean()), float(wh[1].mean()), "max", float(wh[0].max()), float(wh[1].max()))
wh = (small[:, 3] - small[:, 1]), (small[:, 4] - small[:, 2])
print("small roi w/h mean", float(wh[0].mean()), float(wh[1].mean()))
