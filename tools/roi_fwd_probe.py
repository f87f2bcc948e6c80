"""Developer tool: RoIPool forward (with argmax) on the config-3 shape, synthetic and RPN-made rois, L2 flushed between
launches.  Prints microseconds per launch."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from faster_rcnn_pytorch_b200 import ops, region, synth
dev = torch.device("cuda:0")
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


for tag, B, C, fh, fw, per in (("cfg3", 16, 512, 37, 62, 128), ("cfg4", 8, 512, 50, 83, 300)):
    feat = torch.from_numpy(synth.features(1, B, C, fh, fw)).to(dev)
    syn = torch.from_numpy(np.concatenate([np.concatenate([np.full((per, 1), b, np.float32), synth.random_rois(10 + b, per, fh, fw, 1)[:, 1:]], 1) for b in range(B)])).to(dev)
    hw = (fh * 16, fw * 16)
    n = synth.num_anchors(hw)
    rs = np.random.RandomState(77)
    lg = torch.from_numpy(rs.standard_normal((B, n, 2)).astype(np.float32)).to(dev)
    rg = torch.from_numpy((rs.standard_normal((B, n, 4)) * 0.2).astype(np.float32)).to(dev)
    pr, pc = region.rpn_proposals(lg, rg, image_hw=hw, mode="train")
    boxes = pr[:, :per].cpu().numpy() * np.array([fw, fh, fw, fh], np.float32)
    rpn = torch.from_numpy(np.concatenate([np.concatenate([np.full((per, 1), b, np.float32), boxes[b]], 1) for b in range(B)])).to(dev)
    for name, r in (("synthetic", syn), ("rpn", rpn)):
        a = timeit(lambda: ops.roi_pool_forward(feat, r))
        print(f"{tag} {name}: {a:.1f} us", flush=True)
