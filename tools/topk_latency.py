"""Developer tool: device time of frr_topk_desc_opt (graph replay of 20 calls) at batch 1 / 8 / 64 for the three proposal
shapes, with the CTAs per image chosen automatically (ctas_per_image 0) and with one CTA per image (ctas_per_image 1)."""
import os, sys
sys.path.insert(0, os.getcwd())
import numpy as np, torch
from faster_rcnn_pytorch_b200 import ops, synth, _lib
dev = torch.device("cuda:0")
lib = _lib.load()
for HW, k in (((608, 1008), 12000), ((600, 1000), 6000), ((800, 1333), 6000)):
    for B in (1, 8, 64):
        ins = [synth.rpn_head_outputs(2000 + i, HW) for i in range(min(B, 4))]
        reg = torch.from_numpy(np.stack([ins[i % len(ins)][1] for i in range(B)])).to(dev)
        sc = torch.from_numpy(np.stack([ins[i % len(ins)][2] for i in range(B)])).to(dev)
        boxes, scores, valid = ops.rpn_decode(reg, sc, image_hw=HW)
        N = scores.shape[1]
        oi = torch.empty((B, k), dtype=torch.int32, device=dev); oc = torch.empty((B,), dtype=torch.int32, device=dev)
        for cpi in (0, 1):
            def run():
                st = torch.cuda.current_stream().cuda_stream
                _lib.check(lib.frr_topk_desc_opt(scores.data_ptr(), valid.data_ptr(), None, B, N, k, None, oi.data_ptr(), None,
                                                 None, oc.data_ptr(), cpi, st), "topk")
            for _ in range(3): run()
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize()
            with torch.cuda.graph(g):
                for _ in range(20): run()
            g.replay(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
            print(f"HW={HW} k={k} B={B} ctas_per_image={cpi}: {e0.elapsed_time(e1)/20*1e3:.1f} us", flush=True)
