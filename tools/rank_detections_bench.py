"""Cost of the score-ranked evaluation hand-off: class_nms + pack_detections(rank="score") against class_nms +
pack_detections(rank="class"), at the config 4 shape of SURVEY §8d (B = 8 images, R = 300 rois, C = 81 classes) and
score thresholds 0.05 (the reference default) and 0.005 (the dense stress case).

Inputs: seeded head outputs decoded by decode_classwise, as in FRCNN.predict.  Each form is captured into a CUDA graph of
--reps back-to-back calls; the graphs of all forms are replayed in turn (A, B, C, A, B, C, ...) --steps times after
--warmup replays, each replay timed with CUDA events, and the median time per call is reported.  prob and boxes of a
batch (3.9 MB) stay in the 126 MB L2 between calls, as they do in the real pipeline, where decode_classwise has just
written them.  The pack kernels alone are timed the same way on the class_nms output.  The card name and power limit
are read in the same run and printed with the numbers.  One JSON line per (threshold, form).

    python tools/rank_detections_bench.py [--steps 50] [--warmup 5] [--reps 20] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

from faster_rcnn_pytorch_b200 import ops, synth  # noqa: E402

B, R, C = 8, 300, 81
FORMS = {  # name -> pack_detections arguments
    "class": dict(max_det=100, rank="class"),
    "score": dict(max_det=100, rank="score"),
    "score_per_class_100": dict(max_det=100, rank="score", per_class_max=100),
}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(device=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.stdout else None)


def head_batch(dev):
    heads = [synth.head_outputs(4000 + i, R, C) for i in range(B)]
    rois = np.concatenate([synth.random_boxes(4100 + i, R)[0] for i in range(B)])
    cls = torch.from_numpy(np.concatenate([h[0] for h in heads])).to(dev)
    reg = torch.from_numpy(np.concatenate([h[1] for h in heads])).to(dev)
    prob, boxes = ops.decode_classwise(cls, reg, torch.from_numpy(rois).to(dev), C)
    return prob.view(B, R, C), boxes.view(B, R, 4 * C)


def capture(fn, reps, dev):
    fn()
    torch.cuda.synchronize(dev)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    return g


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("rank_detections_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    info = card()
    print(json.dumps(info), flush=True)
    prob, boxes = head_batch(dev)
    ws = ops.pack_ranked_workspace(B, R * (C - 1), 100, dev)
    lines = []
    for thres in (0.05, 0.005):
        det = ops.class_nms(prob, boxes, C, score_thres=thres, iou_thr=0.3)
        counts = det[3].cpu().tolist()
        graphs = {}
        for name, kw in FORMS.items():
            def pack(kw=kw):
                return ops.pack_detections(*det, workspace=ws, **kw)

            def nms_pack(kw=kw):
                d = ops.class_nms(prob, boxes, C, score_thres=thres, iou_thr=0.3)
                return ops.pack_detections(*d, workspace=ws, **kw)
            graphs[(name, "class_nms+pack")] = capture(nms_pack, a.reps, dev)
            graphs[(name, "pack")] = capture(pack, a.reps, dev)
        times = {k: [] for k in graphs}
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in graphs]
        for step in range(a.warmup + a.steps):
            for (k, g), (e0, e1) in zip(graphs.items(), ev):
                e0.record()
                g.replay()
                e1.record()
            torch.cuda.synchronize(dev)
            if step >= a.warmup:
                for k, (e0, e1) in zip(graphs, ev):
                    times[k].append(e0.elapsed_time(e1) * 1e3 / a.reps)
        for (name, what), t in times.items():
            rec = dict(B=B, R=R, C=C, score_thres=thres, detections_per_image=counts, form=name, timed=what,
                       us_per_call_median=round(statistics.median(t), 2), us_per_call_min=round(min(t), 2),
                       us_per_call_max=round(max(t), 2), replays=a.steps, calls_per_replay=a.reps, **info)
            print(json.dumps(rec), flush=True)
            lines.append(rec)
    if a.out:
        with open(a.out, "a") as fh:
            for rec in lines:
                fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
