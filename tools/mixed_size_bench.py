"""Mixed-size batches vs bucketing vs per-image modules: the VGG region stage on a VOC-like size mix.

Half the images are 600 x 800 (H x W), half 800 x 600; stride 16.  Three ways to run them, at B = 16 and 64 images:

  sized     one batch padded to 800 x 800 (a 50 x 50 grid), per-image sizes in an int32 [B,2] device tensor, one CUDA
            graph per stage;
  bucketed  two uniform batches of B/2 (37 x 50 and 50 x 37 grids), one CUDA graph per bucket and stage;
  modules   the single-image ``modules.*`` drop-ins, one image at a time (they synchronise with the host per image).

Stages (models/model.py:310-335 and :346-366):
  infer  proposals in test mode (6000 -> 300) + roi scaling + RoIPool 7x7 forward on a 512-channel map;
  train  proposals in train mode (12000 -> 2000) + both target makers (sampling on the device for the batched forms,
         the host torch.randperm path for the modules) + RoIPool forward with argmax + its backward.

Time per batch from CUDA events over --steps replays (or loops) after --warmup, inputs seeded.  The feature maps of a
B = 64 batch are 327 MB (sized) / 242 MB (bucketed), larger than the 126 MB L2.  The card name and power limit are read
in the same run and printed with the numbers.  One JSON line per (stage, B, form) on stdout and in --out.

    python tools/mixed_size_bench.py [--steps 30] [--warmup 5] [--batches 16,64] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

from faster_rcnn_pytorch_b200 import modules, ops, region, targets  # noqa: E402

STRIDE, A, C = 16, 9, 512
SIZES = ((600, 800), (800, 600))
MAX_HW = (800, 800)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(device=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.stdout else None)


def inputs(B, hw_grid, sizes, seed, dev):
    """head outputs on the grid (padding cells hold NaN, as a padded conv output might), features, gt"""
    gh, gw = hw_grid
    g = torch.Generator().manual_seed(seed)
    N = gh * gw * A
    cls = torch.randn((B, N, 2), generator=g)
    reg = torch.randn((B, N, 4), generator=g) * 0.2
    feat = torch.randn((B, C, gh, gw), generator=g)
    for b, (h, w) in enumerate(sizes):
        m = torch.ones((gh, gw), dtype=torch.bool)
        m[:h // STRIDE, :w // STRIDE] = False
        cls.view(B, gh, gw, A, 2)[b][m] = float("nan")
        reg.view(B, gh, gw, A, 4)[b][m] = float("nan")
        feat[b][:, m] = 0.0
    rs = np.random.RandomState(seed)
    G = 8
    xy1 = rs.uniform(0.0, 0.7, (B, G, 2))
    wh = rs.uniform(0.05, 0.3, (B, G, 2))
    gt = torch.from_numpy(np.concatenate([xy1, xy1 + wh], axis=2).astype(np.float32))
    gtc = torch.from_numpy(rs.randint(1, G + 1, B).astype(np.int32))
    lab = torch.from_numpy(rs.randint(0, 20, (B, G)).astype(np.int64))
    return [t.to(dev) for t in (cls, reg, feat, gt, gtc, lab)]


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


class Batch:
    """one batch (uniform or sized) with its infer and train steps captured into CUDA graphs"""

    def __init__(self, B, hw, sizes, seed, dev, sized):
        self.hw_t = torch.tensor(sizes, dtype=torch.int32, device=dev) if sized else None
        grid = (hw[0] // STRIDE, hw[1] // STRIDE)
        self.cls, self.reg, self.feat, self.gt, self.gtc, self.lab = inputs(B, grid, sizes, seed, dev)
        N = grid[0] * grid[1] * A
        self.infer = region.InferPlan(B, hw, 21, dev)
        self.prop = region.ProposalPlan(B, N, dev, image_hw=hw, mode="train")
        self.train = region.TrainPlan(B, hw, dev)
        self.g_infer, _ = self.infer.capture_pool(self.feat, self.cls, self.reg, image_hw=self.hw_t)
        self.g_prop = self.prop.capture(self.cls, self.reg, self.hw_t)
        self.prop.run(self.cls, self.reg, image_hw=self.hw_t)
        self.g_tp, (_, pooled) = self.train.capture_targets_and_pool(self.feat, self.gt, self.lab, self.prop.rois,
                                                                      self.prop.count, image_hw=self.hw_t)
        self.go = torch.ones_like(pooled)
        self.g_bwd, _ = self.train.capture_pool_backward(self.go)

    def infer_step(self):
        self.g_infer.replay()

    def train_step(self):
        self.g_prop.replay()
        self.g_tp.replay()
        self.g_bwd.replay()


def modules_steps(B, sizes, seed, dev):
    """the single-image drop-ins, image by image, on each image's own unpadded inputs"""
    per = []
    for b, hw in enumerate(sizes):
        grid = (hw[0] // STRIDE, hw[1] // STRIDE)
        cls, reg, feat, gt, gtc, lab = inputs(1, grid, [hw], seed + b, dev)
        per.append((hw, grid, ops.anchors(hw, dev), cls[0], reg[0], feat, gt[0, :int(gtc[0])], lab[0, :int(gtc[0])]))
    rp, rpn_t, frc_t, pool = modules.RegionProposal(), modules.RPNTargetMaker(), modules.FastRcnnTargetMaker(), \
        modules.RoIPool((7, 7), 1.0)

    def scale(rois, grid):
        return rois * torch.tensor([grid[1], grid[0], grid[1], grid[0]], dtype=torch.float32, device=dev)

    def infer():
        for hw, grid, anc, cls, reg, feat, gt, lab in per:
            rois = rp(cls, reg, anc, "test")
            pool(feat, [scale(rois, grid)])

    def train():
        for hw, grid, anc, cls, reg, feat, gt, lab in per:
            rois = rp(cls, reg, anc, "train")
            rpn_t(gt, anc)
            _, _, srois = frc_t([gt], [lab], rois)
            f = feat.detach().requires_grad_(True)
            out = pool(f, [scale(srois, grid)])
            out.backward(torch.ones_like(out))
    return infer, train


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batches", default="16,64")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mixed_size_bench needs a CUDA device: there is nothing to measure without one")
    dev = torch.device("cuda:0")
    info = card()
    lines = []
    for B in (int(x) for x in args.batches.split(",")):
        half = B // 2
        sizes = [SIZES[i % 2] for i in range(B)]                      # interleaved 600x800 / 800x600
        torch.manual_seed(0)
        sized = Batch(B, MAX_HW, sizes, 1, dev, True)
        buckets = [Batch(half, hw, [hw] * half, 2 + i, dev, False) for i, hw in enumerate(SIZES)]
        m_infer, m_train = modules_steps(B, sizes, 10, dev)
        forms = {
            "sized": (sized.infer_step, sized.train_step),
            "bucketed": (lambda: [bk.infer_step() for bk in buckets], lambda: [bk.train_step() for bk in buckets]),
            "modules": (m_infer, m_train),
        }
        for stage, k in (("infer", 0), ("train", 1)):
            for form, fns in forms.items():
                steps = args.steps if form != "modules" else max(3, args.steps // 5)
                ms = timed(fns[k], steps, args.warmup)
                line = dict(stage=stage, B=B, form=form, ms_per_batch=round(ms, 4),
                            images_per_s=round(B / ms * 1e3, 1), steps=steps, sizes="600x800/800x600",
                            padded_to="800x800" if form == "sized" else None, **info)
                print(json.dumps(line), flush=True)
                lines.append(line)
        del sized, buckets
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
