"""Developer tool: the deterministic RoIPool / RoIAlign backward (torch.use_deterministic_algorithms) next to the default
kernels and torchvision's CUDA backward, at config 3 (16 x 512 x 37 x 62, 2048 rois), on the 50 x 83 map of an
800 x 1333 image and for MultiScaleRoIAlign forward + backward at the shapes of tools/msroialign_profile.py.

    python tools/roi_bwd_det_profile.py [out.txt]

CUDA events around each call, a 256 MB buffer overwritten before every timed pass (nothing stays in the 126 MB L2),
mean of 20 passes after 3 warm-ups.  Bytes are algorithmic: grad_out (+ argmax) read once, grad_in written once (the
MultiScaleRoIAlign rows add the forward's feature reads and output write)."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torchvision  # noqa: F401  (registers torch.ops.torchvision)

from faster_rcnn_pytorch_b200 import ops, synth

dev = torch.device("cuda:0")
flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


def timeit(fn, reps=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / reps * 1e3


def row(name, us, nbytes):
    say(f"  {name:<34s} {us:9.1f} us  {nbytes / 1e6:8.1f} MB  {nbytes / us / 1e3:7.1f} GB/s")


def rpn_rois(seed, K, B, fh, fw):
    b, _ = synth.random_boxes(seed, K)
    return np.concatenate([np.repeat(np.arange(B), K // B)[:, None], b * np.array([fw, fh, fw, fh])], 1).astype(np.float32)


def single_level(label, B, C, fh, fw, K):
    say(f"{label}: B {B}, C {C}, {fh} x {fw}, K {K}, RPN-sized rois")
    feat = torch.from_numpy(synth.features(1, B, C, fh, fw)).to(dev)
    rois = torch.from_numpy(rpn_rois(2, K, B, fh, fw)).to(dev)
    go = torch.randn((K, C, 7, 7), device=dev)
    _, arg = ops.roi_pool_forward(feat, rois)
    _, arg_tv = torch.ops.torchvision.roi_pool(feat, rois, 1.0, 7, 7)
    shape = (B, C, fh, fw)
    rows = K * C * 49 * 4
    gin = B * C * fh * fw * 4
    say(f"  RoIPool backward (default kernel: {ops.roi_variant('roi_pool_bwd', K, B, C, fh, fw)['kernel']})")
    row("default", timeit(lambda: ops.roi_pool_backward(go, arg, rois, shape, deterministic=False)), 2 * rows + gin)
    row("deterministic", timeit(lambda: ops.roi_pool_backward(go, arg, rois, shape, deterministic=True)), 2 * rows + gin)
    row("torchvision CUDA", timeit(lambda: torch.ops.torchvision._roi_pool_backward(go, rois, arg_tv, 1.0, 7, 7, B, C, fh,
                                                                                    fw)), 2 * rows + gin)
    say(f"  RoIAlign backward, sampling 2 (default kernel: {ops.roi_variant('roi_align_bwd', K, B, C, fh, fw)['kernel']})")
    row("default", timeit(lambda: ops.roi_align_backward(go, rois, shape, 1.0, 2, deterministic=False)), rows + gin)
    row("deterministic", timeit(lambda: ops.roi_align_backward(go, rois, shape, 1.0, 2, deterministic=True)), rows + gin)
    row("torchvision CUDA", timeit(lambda: torch.ops.torchvision._roi_align_backward(go, rois, 1.0, 7, 7, B, C, fh, fw, 2,
                                                                                     False)), rows + gin)
    # the same sums in a different order: the deterministic result against the default one
    a = ops.roi_align_backward(go, rois, shape, 1.0, 2, deterministic=False)
    d = ops.roi_align_backward(go, rois, shape, 1.0, 2, deterministic=True)
    say(f"  RoIAlign |det - default| max / max|grad| = {float((a - d).abs().max() / d.abs().max()):.2e}")


def multiscale():
    B, C, hw, per = 2, 256, (800, 1344), 512
    say(f"MultiScaleRoIAlign forward + backward: B {B}, C {C}, {hw[0]} x {hw[1]} input, strides 4-32, {per} rois per image")
    rs = np.random.RandomState(5)
    feats = [torch.from_numpy(rs.standard_normal((B, C, hw[0] // s, hw[1] // s)).astype(np.float32)).to(dev)
             for s in (4, 8, 16, 32)]
    side = np.exp(rs.uniform(np.log(16), np.log(600), B * per))
    ar = np.exp(rs.uniform(-0.7, 0.7, B * per))
    w, h = side * np.sqrt(ar), side / np.sqrt(ar)
    cx, cy = rs.uniform(0, hw[1], B * per), rs.uniform(0, hw[0], B * per)
    x1, y1 = np.clip(cx - w / 2, 0, hw[1] - 2), np.clip(cy - h / 2, 0, hw[0] - 2)
    x2, y2 = np.clip(cx + w / 2, x1 + 1, hw[1]), np.clip(cy + h / 2, y1 + 1, hw[0])
    boxes = [torch.from_numpy(np.stack([x1, y1, x2, y2], 1)[b * per:(b + 1) * per].astype(np.float32)).to(dev)
             for b in range(B)]
    shapes = [hw] * B
    fg = [f.clone().requires_grad_(True) for f in feats]
    go = torch.randn((B * per, C, 7, 7), device=dev)
    tv = torchvision.ops.MultiScaleRoIAlign(["0", "1", "2", "3"], 7, 2)
    nbytes = 2 * sum(f.numel() for f in feats) * 4 + 2 * go.numel() * 4

    def ours(det):
        def fn():
            prev = torch.are_deterministic_algorithms_enabled()
            torch.use_deterministic_algorithms(det)
            try:
                ops.multiscale_roi_align(fg, boxes, shapes, 7, 2).backward(go)
            finally:
                torch.use_deterministic_algorithms(prev)
        return fn

    row("default", timeit(ours(False)), nbytes)
    row("deterministic", timeit(ours(True)), nbytes)
    row("torchvision CUDA", timeit(lambda: tv({str(i): f for i, f in enumerate(fg)}, boxes, shapes).backward(go)), nbytes)


def main():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    say(f"device: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit: {q[0] if q else 'n/a'}")
    single_level("config 3", 16, 512, 37, 62, 2048)
    single_level("800 x 1333 image", 8, 512, 50, 83, 2400)
    multiscale()
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
