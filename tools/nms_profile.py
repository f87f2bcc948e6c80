"""Developer tool: bucketed NMS kernel timing over its per-call settings on the config-2 workload (GPU box)."""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from faster_rcnn_pytorch_b200 import ops, synth

HW = (608, 1008)
dev = torch.device("cuda:0")
B = int(os.environ.get("NMS_B", "64"))
ins = [synth.rpn_head_outputs(2000 + i, HW) for i in range(B)]
reg = torch.from_numpy(np.stack([x[1] for x in ins])).to(dev)
sc = torch.from_numpy(np.stack([x[2] for x in ins])).to(dev)
boxes, scores, valid = ops.rpn_decode(reg, sc, image_hw=HW)
top = ops.topk_desc(scores, 12000, valid=valid, boxes=boxes)
tb, tc = top["boxes"], top["count"]


def run(bx, cnt, S, threads, tune, reps=20):
    for _ in range(3):
        ops.nms_sorted(bx, 0.7, max_keep=2000, counts=cnt, cluster_size=S, threads=threads, unit_boxes=True, **tune)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        ops.nms_sorted(bx, 0.7, max_keep=2000, counts=cnt, cluster_size=S, threads=threads, unit_boxes=True, **tune)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    keep, c, _ = ops.nms_sorted(bx, 0.7, max_keep=2000, counts=cnt, cluster_size=S, threads=threads, unit_boxes=True, **tune)
    out = {"B": bx.shape[0], "S": S, "threads": threads, "us": round(ms * 1e3, 1), "kept": int(c[0]),
           "last_keep_pos": int(keep[0, int(c[0]) - 1])}
    print(json.dumps(out), flush=True)


one, onec = tb[:1].contiguous(), tc[:1].contiguous()
for first, largest, n1, n2 in ((512, 2048, 4, 4), (512, 2048, 8, 8), (512, 2048, 2, 2), (512, 2048, 1, 1), (512, 2048, 8, 4),
                               (512, 2048, 16, 8), (1024, 2048, 4, 4), (256, 2048, 4, 4), (512, 1536, 4, 4), (768, 2048, 4, 4)):
    tune = dict(first_chunk=first, max_chunk=largest, lanes_screen=n1, lanes_pairs=n2)
    print(json.dumps(tune), flush=True)
    for threads, S in ((1024, 2), (1024, 1), (1024, 4)):
        run(tb, tc, S, threads, tune)
    for threads, S in ((1024, 16), (512, 16), (1024, 8)):
        run(one, onec, S, threads, tune, reps=50)
