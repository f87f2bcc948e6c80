"""Golden fixtures for the long-roi-list RoIPool forward test (tests/test_gpu_roi.py).

    python tests/golden/make_golden_roi_long.py [OUT.npz]

Runs torchvision's RoIPool (torch.ops.torchvision.roi_pool, 7x7, scale 1.0; its CUDA kernel when a GPU is present, else
its CPU kernel) on the test's seeded inputs and stores, per case, the sha256 of the max and argmax arrays of the unmasked
rois, their shape, and the values at a seeded sample of positions (tests/golden/roi_long.npz): the outputs themselves are
several MB per case.  The stored file was made with torchvision 0.26.0's CPU kernel, whose max and argmax on these inputs
are also bit-equal to the C oracle's (oracle/c/region_oracle.c).
"""
import hashlib
import os
import sys

import numpy as np
import torch
import torchvision  # noqa: F401  (registers torch.ops.torchvision)

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path.insert(0, TESTS)
sys.path.insert(0, os.path.dirname(TESTS))
from faster_rcnn_pytorch_b200 import synth  # noqa: E402
from test_gpu_roi import LONG_ROI_CASES, LONG_ROI_SHAPE, _mixed_rois  # noqa: E402

SAMPLE = 4096


def sha(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


def main(path):
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    C, fh, fw = LONG_ROI_SHAPE
    g = {}
    for K, B, _ in LONG_ROI_CASES:
        feat = torch.from_numpy(synth.features(710, B, C, fh, fw)).to(dev)
        rois5 = _mixed_rois(711, K, fh, fw, B, small_frac=0.2)
        keep = rois5[:, 0] >= 0
        out, arg = torch.ops.torchvision.roi_pool(feat, torch.from_numpy(rois5[keep]).to(dev), 1.0, 7, 7)
        out, arg = out.cpu().numpy(), arg.cpu().numpy().astype(np.int32)
        idx = np.sort(np.random.RandomState(K).choice(out.size, SAMPLE, replace=False))
        key = f"{K}_{B}"
        g[f"{key}_shape"] = np.asarray(out.shape, np.int64)
        g[f"{key}_out_sha"], g[f"{key}_argmax_sha"] = sha(out), sha(arg)
        g[f"{key}_idx"] = idx
        g[f"{key}_out_sample"], g[f"{key}_argmax_sample"] = out.reshape(-1)[idx], arg.reshape(-1)[idx]
    np.savez_compressed(path, **g)
    print(path, os.path.getsize(path), "torchvision", torchvision.__version__, dev)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "roi_long.npz"))
