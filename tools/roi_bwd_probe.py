"""Developer tool: RoIPool backward on rois of a controlled size (cells) -- ours vs torchvision's CUDA kernel."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, torchvision
from faster_rcnn_pytorch_b200 import ops, synth
dev = torch.device("cuda:0")
B, C, fh, fw, per = (8, 512, 50, 83, 300) if "cfg4" in sys.argv else (16, 512, 37, 62, 128)
print("shape", (B, C, fh, fw, per), flush=True)
K = B * per
feat = torch.from_numpy(synth.features(1, B, C, fh, fw)).to(dev)
go = torch.randn((K, C, 7, 7), device=dev)
flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)


def timeit(fn, reps=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / reps * 1e3


for lo, hi in ((8, 30), (7, 14), (3, 7), (1, 3), (1, 30)):
    rs = np.random.RandomState(5)
    w = rs.uniform(lo, hi, K); h = rs.uniform(lo, min(hi, fh - 1), K)
    x1 = rs.uniform(0, fw - w); y1 = rs.uniform(0, fh - h)
    rois = np.stack([np.repeat(np.arange(B), per), x1, y1, x1 + w, y1 + h], 1).astype(np.float32)
    r = torch.from_numpy(rois).to(dev)
    out, arg = ops.roi_pool_forward(feat, r)
    us = timeit(lambda: ops.roi_pool_backward(go, arg, r, feat.shape))
    o2, a2 = torch.ops.torchvision.roi_pool(feat, r, 1.0, 7, 7)
    tv = timeit(lambda: torch.ops.torchvision._roi_pool_backward(go, r, a2, 1.0, 7, 7, B, C, fh, fw))
    print(f"roi side {lo}-{hi} cells: ours {us:.1f} us, torchvision {tv:.1f} us", flush=True)
