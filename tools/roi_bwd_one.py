"""Developer tool: RoIPool backward at the config-3 / config-4 shape on rois of a controlled size -- also the
single-launch target for ncu.

    [ROI_LO=8 ROI_HI=30] python tools/roi_bwd_one.py [cfg4]
"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from faster_rcnn_pytorch_b200 import ops, synth
dev = torch.device("cuda:0")
B, C, fh, fw, per = (8, 512, 50, 83, 300) if "cfg4" in sys.argv else (16, 512, 37, 62, 128)
K = B * per
feat = torch.from_numpy(synth.features(1, B, C, fh, fw)).to(dev)
go = torch.randn((K, C, 7, 7), device=dev)
rs = np.random.RandomState(5)
lo, hi = float(os.environ.get("ROI_LO", "8")), float(os.environ.get("ROI_HI", "30"))
w = rs.uniform(lo, hi, K); h = rs.uniform(lo, min(hi, fh - 1), K)
x1 = rs.uniform(0, fw - w); y1 = rs.uniform(0, fh - h)
r = torch.from_numpy(np.stack([np.repeat(np.arange(B), per), x1, y1, x1 + w, y1 + h], 1).astype(np.float32)).to(dev)
out, arg = ops.roi_pool_forward(feat, r)
gin = ops.roi_pool_backward(go, arg, r, feat.shape)
torch.cuda.synchronize()
reps = 5
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(reps):
    gin = ops.roi_pool_backward(go, arg, r, feat.shape)
e1.record()
torch.cuda.synchronize()
print(f"roi side {lo}-{hi} shape {(B, C, fh, fw, per)}: {e0.elapsed_time(e1) / reps * 1e3:.1f} us per launch")
