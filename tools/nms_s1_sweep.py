"""Developer tool: bucketed NMS with ONE CTA per image (the throughput geometry) over the per-call settings of frr_nms_sorted."""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from faster_rcnn_pytorch_b200 import ops, synth
HW = (608, 1008)
dev = torch.device("cuda:0")
B = 64
ins = [synth.rpn_head_outputs(2000 + i, HW) for i in range(B)]
reg = torch.from_numpy(np.stack([x[1] for x in ins])).to(dev)
sc = torch.from_numpy(np.stack([x[2] for x in ins])).to(dev)
boxes, scores, valid = ops.rpn_decode(reg, sc, image_hw=HW)
top = ops.topk_desc(scores, 12000, valid=valid, boxes=boxes)
tb, tc = top["boxes"], top["count"]
ref = None
for S in (1, 2):
    for first in (1024,):
        for largest in (2048,):
            for n1, n2 in ((1, 4), (2, 4), (2, 8), (1, 8), (4, 4), (2, 16), (8, 4)):
                tune = dict(first_chunk=first, max_chunk=largest, lanes_screen=n1, lanes_pairs=n2)
                for _ in range(2):
                    keep, c, _r = ops.nms_sorted(tb, 0.7, max_keep=2000, counts=tc, cluster_size=S, unit_boxes=True, **tune)
                torch.cuda.synchronize()
                if ref is None:
                    ref = keep.clone()
                assert torch.equal(keep, ref)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(10):
                    ops.nms_sorted(tb, 0.7, max_keep=2000, counts=tc, cluster_size=S, unit_boxes=True, **tune)
                e1.record(); torch.cuda.synchronize()
                print(json.dumps({"S": S, "first": first, "largest": largest, "lanes": [n1, n2], "us": round(e0.elapsed_time(e1) * 100, 1)}), flush=True)
