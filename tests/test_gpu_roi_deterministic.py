"""Deterministic RoIPool / RoIAlign backward (frr_roi_*_bwd_deterministic, torch.use_deterministic_algorithms): every
gradient array-equal to torchvision's CPU backward (goldens, and the CPU oracle at production shapes for the territory of
every default kernel), identical across streams, graph replay and concurrent work, and selected by PyTorch's switch."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import REPO, golden
from faster_rcnn_pytorch_b200 import modules, ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BWD_KERNELS = ("roi_pool_bwd_color_kernel", "roi_pool_bwd_tail_kernel", "roi_align_bwd_fast_kernel",
               "roi_align_bwd_stream_kernel", "roi_bwd_planes_kernel", "roi_bwd_direct_kernel", "roi_bwd_det_kernel")


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def same(got, want):
    """bit-equal, NaN positions included"""
    got = got.cpu().numpy() if isinstance(got, torch.Tensor) else got
    assert got.shape == want.shape and got.dtype == want.dtype
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    assert np.array_equal(got[ok].view(np.uint32), want[ok].view(np.uint32))


@pytest.fixture
def det_flag():
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev)


def live(rois5, B):
    b = rois5[:, 0].astype(np.int64)
    return (b >= 0) & (b < B) & (rois5[:, 0] == b)


def check_pool(oracle, feat, rois5, go, scale=1.0, osz=(7, 7), channels_last=False):
    B = feat.shape[0]
    f = dev(feat)
    if channels_last:
        f = f.contiguous(memory_format=torch.channels_last)
    _, arg = ops.roi_pool_forward(f, dev(rois5), osz, scale)
    gin = ops.roi_pool_backward(dev(go), arg, dev(rois5), feat.shape, scale, channels_last, deterministic=True)
    assert gin.is_contiguous(memory_format=torch.channels_last if channels_last else torch.contiguous_format)
    m = live(rois5, B)
    want = oracle.roi_pool_backward(go[m], arg.cpu().numpy()[m], rois5[m], feat.shape)
    same(gin, want)
    return gin


def check_align(oracle, shape, rois5, go, scale=1.0, sr=2, aligned=False, channels_last=False):
    B = shape[0]
    gin = ops.roi_align_backward(dev(go), dev(rois5), shape, scale, sr, aligned, channels_last, deterministic=True)
    m = live(rois5, B)
    want = oracle.roi_align_backward(go[m], rois5[m], shape, go.shape[2:], scale, sr, aligned)
    same(gin, want)
    return gin


def grad_out(seed, K, C, osz=(7, 7)):
    return np.random.RandomState(seed).standard_normal((K, C) + tuple(osz)).astype(np.float32)


def rpn_rois(seed, K, B, fh, fw, scale=1.0):
    """proposal-like boxes (clustered, 2-30 % of the image side), per-image blocks, in map coordinates / scale"""
    b, _ = synth.random_boxes(seed, K)
    r = np.concatenate([np.repeat(np.arange(B), -(-K // B))[:K, None], b * np.array([fw, fh, fw, fh]) / scale], 1)
    return r.astype(np.float32)


# ---------------------------------------------------------------------------------------------------------------------
# goldens (torchvision CPU)
# ---------------------------------------------------------------------------------------------------------------------
CASES = [("a", 500, 1, 8, 37, 62, 64), ("b", 501, 2, 16, 10, 14, 40), ("c", 502, 1, 4, 5, 6, 30)]


@pytest.mark.parametrize("name,seed,B,C,fh,fw,K", CASES)
@pytest.mark.parametrize("channels_last", [False, True])
def test_goldens_bit_exact(name, seed, B, C, fh, fw, K, channels_last):
    g = golden("roi")
    feat = dev(synth.features(seed, B, C, fh, fw))
    if channels_last:
        feat = feat.contiguous(memory_format=torch.channels_last)
    rois5 = dev(synth.random_rois(seed + 1, K, fh, fw, B))
    go = dev(np.random.RandomState(seed + 2).standard_normal((K, C, 7, 7)).astype(np.float32))
    _, arg = ops.roi_pool_forward(feat, rois5)
    same(ops.roi_pool_backward(go, arg, rois5, feat.shape, channels_last=channels_last, deterministic=True),
         g[f"{name}_pool_gin"])
    for scale in (1.0, 0.5):
        gin = ops.roi_align_backward(go, rois5, feat.shape, scale, 2, False, channels_last, deterministic=True)
        same(gin, g[f"{name}_align_gin_{scale}"])


@pytest.mark.parametrize("tag,shapes", [("hw", [(256, 320)] * 2), ("wh_like_reference", [(320, 256)] * 2)])
@pytest.mark.parametrize("channels_last", [False, True])
def test_multiscale_goldens_through_autograd(det_flag, tag, shapes, channels_last):
    g = golden("msroialign")
    feats_np, rois5 = synth.pyramid_inputs(image_hw=(256, 320))
    feats = [dev(f) for f in feats_np]
    if channels_last:
        feats = [f.contiguous(memory_format=torch.channels_last) for f in feats]
    feats = [f.requires_grad_(True) for f in feats]
    out = modules.MultiScaleRoIAlign(["0", "1", "2", "3"], 7, 2)({str(i): f for i, f in enumerate(feats)}, dev(rois5),
                                                                 shapes)
    out.backward(dev(g["grad_out"]))
    for i, f in enumerate(feats):
        same(f.grad, g[f"{tag}_gin{i}"])


# ---------------------------------------------------------------------------------------------------------------------
# CPU oracle at production shapes: one case per territory of every default backward kernel
# ---------------------------------------------------------------------------------------------------------------------
def test_pool_config3_rpn_rois_post_relu(oracle):
    """16 x 512 x 37 x 62, K 2048 (colour-class + tail kernels by default), argmax ties on whole zero windows"""
    B, C, fh, fw, K = 16, 512, 37, 62, 2048
    feat = np.maximum(synth.features(900, B, C, fh, fw), 0.0)
    check_pool(oracle, feat, rpn_rois(901, K, B, fh, fw), grad_out(902, K, C))


@pytest.mark.parametrize("channels_last", [False, True])
def test_pool_and_align_50x83(oracle, channels_last):
    """800 x 1333 map, K 2400: the tail-only RoIPool kernel and the streaming RoIAlign kernel by default"""
    B, C, fh, fw, K = 8, 64, 50, 83, 2400
    feat = synth.features(910, B, C, fh, fw)
    rois5 = rpn_rois(911, K, B, fh, fw)
    go = grad_out(912, K, C)
    check_pool(oracle, feat, rois5, go, channels_last=channels_last)
    check_align(oracle, feat.shape, rois5, go, channels_last=channels_last)


def test_align_fpn_level0_levelmapper_masked(oracle):
    """200 x 336 FPN level 0 at C 256 (planes do not fit shared memory: the direct atomic kernel by default), rois of the
    other levels masked the way MultiScaleRoIAlign masks them"""
    B, C, fh, fw, K = 2, 256, 200, 336, 1024
    side = np.exp(np.random.RandomState(920).uniform(np.log(16), np.log(600), K))
    rs = np.random.RandomState(921)
    cx, cy = rs.uniform(0, fw * 4, K), rs.uniform(0, fh * 4, K)
    rois5 = np.stack([rs.randint(0, B, K), cx - side / 2, cy - side / 2, cx + side / 2, cy + side / 2], 1).astype(np.float32)
    lv = oracle.fpn_levels(rois5, 2, 5)
    rois5[lv != 0, 0] = -1
    assert (lv == 0).sum() > 100
    check_align(oracle, (B, C, fh, fw), rois5, grad_out(922, K, C), scale=0.25)


@pytest.mark.parametrize("B,C,fh,fw,K,osz", [
    (2, 20, 37, 62, 300, (7, 7)),     # partial channel group (16 + 4), bwd planes / colour kernels by default
    (3, 7, 4, 90, 120, (7, 7)),       # thin map, odd channel count
    (2, 9, 70, 3, 120, (7, 7)),       # tall thin map
    (2, 24, 30, 40, 200, (3, 5)),     # 3 x 5 bins: the generic plane kernels by default
    (1, 40, 33, 47, 150, (14, 14)),   # 14 x 14 bins
    # bins so many that a ring of 16-channel slots does not fit shared memory: RoIPool 24 x 24 and 28 x 28 and RoIAlign
    # 28 x 28 run with 8 channels per CTA (40 = 5 groups of 8)
    (1, 40, 33, 47, 60, (24, 24)),
    (2, 40, 30, 41, 50, (28, 28)),
    (1, 6, 45, 50, 12, (40, 40)),     # 2 channels per CTA (3 groups)
])
def test_shapes_and_bins(oracle, B, C, fh, fw, K, osz):
    feat = np.maximum(synth.features(930, B, C, fh, fw), 0.0)
    rois5 = synth.random_rois(931, K, fh, fw, B)
    go = grad_out(932, K, C, osz)
    check_pool(oracle, feat, rois5, go, osz=osz)
    for sr, aligned in ((2, False), (0, True), (-1, False), (3, True)):
        check_align(oracle, feat.shape, rois5, go, sr=sr, aligned=aligned)


@pytest.mark.parametrize("sr", [2, 0, -1])
@pytest.mark.parametrize("aligned", [False, True])
def test_align_sampling_and_alignment_at_scale_1_16(oracle, sr, aligned):
    B, C, fh, fw, K = 4, 256, 37, 62, 512
    check_align(oracle, (B, C, fh, fw), rpn_rois(940, K, B, fh, fw, scale=1 / 16), grad_out(941, K, C),
                scale=1 / 16, sr=sr, aligned=aligned)


def test_masked_out_of_range_and_outside_rois(oracle):
    """masked rows, batch index >= B, rois outside the map, an image without rois (its gradient is all +0.0)"""
    B, C, fh, fw, K = 3, 24, 37, 62, 300
    feat = synth.features(950, B, C, fh, fw)
    rois5 = synth.random_rois(951, K, fh, fw, B)
    rois5[:, 0] = np.where(rois5[:, 0] == 2, 0, rois5[:, 0])      # image 2 has no rois
    rois5[::7, 0] = -1
    rois5[3::11, 0] = 3                                           # index >= B
    rois5[5, 1:] = [-40, -30, -20, -10]
    rois5[6, 1:] = [fw + 5, fh + 5, fw + 30, fh + 20]
    rois5[8, 1:] = [fw - 0.6, fh - 0.6, fw + 3, fh + 3]           # last row / column: snapped taps
    go = grad_out(952, K, C)
    for gin in (check_pool(oracle, feat, rois5, go), check_align(oracle, feat.shape, rois5, go, aligned=True)):
        assert torch.equal(gin[2], torch.zeros_like(gin[2])) and not torch.signbit(gin[2]).any()


@pytest.mark.parametrize("sr", [0, -1])
@pytest.mark.parametrize("aligned", [False, True])
def test_align_adaptive_grids_beyond_the_record_capacity(oracle, sr, aligned):
    """adaptive sampling on rois over 16 x 7 map pixels tall / wide: more than 16 samples per bin side, whose records do
    not fit the ring slot and are recomputed where they are used"""
    B, C, fh, fw, K = 2, 16, 60, 80, 40
    rois5 = synth.random_rois(1000, K, fh, fw, B)
    rs = np.random.RandomState(1001)
    big = rs.rand(K) < 0.5
    x1, y1 = rs.uniform(-40, 20, K), rs.uniform(-40, 10, K)
    rois5[big, 1:] = np.stack([x1, y1, x1 + rs.uniform(115, 200, K), y1 + rs.uniform(115, 180, K)], 1)[big]
    assert (rois5[:, 4] - rois5[:, 2] > 16 * 7).sum() >= 10
    check_align(oracle, (B, C, fh, fw), rois5, grad_out(1002, K, C), sr=sr, aligned=aligned)


@pytest.mark.parametrize("sr", [3, -1])
def test_align_division_at_every_magnitude(oracle, sr):
    """grad_out spread over the whole fp32 exponent range, subnormal results included, divided by counts that are not
    powers of two (9 for sampling 3; 1 to 30-odd for adaptive sampling)"""
    B, C, fh, fw, K = 2, 16, 20, 30, 120
    rs = np.random.RandomState(1010)
    e = np.where(rs.rand(K, C, 7, 7) < 0.4, rs.randint(-149, -120, (K, C, 7, 7)), rs.randint(-149, 120, (K, C, 7, 7)))
    go = (rs.choice([-1.0, 1.0], (K, C, 7, 7)) * rs.uniform(1, 2, (K, C, 7, 7)) * np.exp2(e.astype(np.float64)))
    go = go.astype(np.float32)
    assert (np.abs(go) < np.finfo(np.float32).tiny).sum() > 1000
    gin = check_align(oracle, (B, C, fh, fw), synth.random_rois(1011, K, fh, fw, B), go, sr=sr)
    g = np.abs(gin.cpu().numpy())
    assert ((g > 0) & (g < np.finfo(np.float32).tiny)).any()


def test_nan_and_inf_reach_the_same_elements(oracle):
    B, C, fh, fw, K = 2, 16, 20, 30, 80
    feat = synth.features(960, B, C, fh, fw)
    rois5 = synth.random_rois(961, K, fh, fw, B)
    go = grad_out(962, K, C)
    go[3, 2, 1, 4] = np.nan
    go[10, 5, 6, 0] = np.inf
    go[20, 0, 3, 3] = -np.inf
    check_pool(oracle, feat, rois5, go)
    check_align(oracle, feat.shape, rois5, go)
    check_align(oracle, feat.shape, rois5, go, sr=3)


@pytest.mark.parametrize("channels_last", [False, True])
def test_no_rois_gives_zero_gradient(channels_last):
    shape = (2, 12, 9, 11)
    go = torch.zeros((0, 12, 7, 7), device=DEV)
    r = torch.zeros((0, 5), device=DEV)
    a = torch.zeros((0, 12, 7, 7), dtype=torch.int32, device=DEV)
    for gin in (ops.roi_pool_backward(go, a, r, shape, 1.0, channels_last, deterministic=True),
                ops.roi_align_backward(go, r, shape, 1.0, 2, False, channels_last, deterministic=True)):
        assert torch.equal(gin, torch.zeros(shape, device=DEV)) and not torch.signbit(gin).any()


# ---------------------------------------------------------------------------------------------------------------------
# reproducibility
# ---------------------------------------------------------------------------------------------------------------------
def _problem():
    B, C, fh, fw, K = 4, 128, 37, 62, 1024
    feat = dev(synth.features(970, B, C, fh, fw))
    rois5 = dev(rpn_rois(971, K, B, fh, fw))
    go = dev(grad_out(972, K, C))
    _, arg = ops.roi_pool_forward(feat, rois5)
    pool = lambda: ops.roi_pool_backward(go, arg, rois5, feat.shape, deterministic=True)          # noqa: E731
    align = lambda: ops.roi_align_backward(go, rois5, feat.shape, 1.0, 2, deterministic=True)     # noqa: E731
    noise = lambda: (ops.roi_pool_backward(go, arg, rois5, feat.shape, deterministic=False),      # noqa: E731
                     ops.roi_align_backward(go, rois5, feat.shape, 1.0, 2, deterministic=False))
    return pool, align, noise


def test_same_bits_on_two_streams_in_a_graph_and_next_to_other_work():
    pool, align, noise = _problem()
    ref = (pool(), align())
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    res = {}
    for name, s in (("s1", s1), ("s2", s2)):
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            res[name] = (pool(), align())
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):       # warm-up before capture
        pool(), align()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        res["graph"] = (pool(), align())
    graph.replay()
    torch.cuda.synchronize()
    # the default (atomic) backward on another stream at the same time
    s1.wait_stream(torch.cuda.current_stream())
    s2.wait_stream(torch.cuda.current_stream())
    for _ in range(3):
        with torch.cuda.stream(s2):
            noise()
        with torch.cuda.stream(s1):
            res["busy"] = (pool(), align())
    torch.cuda.synchronize()
    for name, (p, a) in res.items():
        assert torch.equal(p, ref[0]) and torch.equal(a, ref[1]), name


# ---------------------------------------------------------------------------------------------------------------------
# selection by torch.use_deterministic_algorithms
# ---------------------------------------------------------------------------------------------------------------------
def backward_kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = {re.sub(r"^void\s+", "", e.name).replace("frr::", "") for e in prof.events()
             if e.device_type == torch.autograd.DeviceType.CUDA}
    return sorted({k for n in names for k in BWD_KERNELS if n.startswith(k)})


VARIANT_KERNELS = {"pool_bwd_color_tail": ["roi_pool_bwd_color_kernel", "roi_pool_bwd_tail_kernel"],
                   "pool_bwd_tail": ["roi_pool_bwd_tail_kernel"], "align_bwd_fast": ["roi_align_bwd_fast_kernel"],
                   "align_bwd_stream": ["roi_align_bwd_stream_kernel"], "bwd_planes": ["roi_bwd_planes_kernel"],
                   "bwd_direct": ["roi_bwd_direct_kernel"]}


def test_flag_selects_the_deterministic_kernels():
    """checked in a child process: its profiler sessions record kernels launched from the autograd engine's thread, and
    the profiler state they leave behind must not reach later tests of this process"""
    r = subprocess.run([sys.executable, "-c", "import test_gpu_roi_deterministic as t; t.check_selection()"],
                       cwd=os.path.dirname(os.path.abspath(__file__)), capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, PYTHONPATH=os.pathsep.join(
                           [os.path.dirname(os.path.abspath(__file__)), REPO, os.environ.get("PYTHONPATH", "")])))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


def check_selection():
    from faster_rcnn_pytorch_b200 import torch_ops  # noqa: F401
    B, C, fh, fw, K = 2, 32, 37, 62, 64
    feat = dev(synth.features(980, B, C, fh, fw))
    rois5 = dev(synth.random_rois(981, K, fh, fw, B))
    feats_np, prois = synth.pyramid_inputs()
    pyr = [dev(f) for f in feats_np]
    go = torch.ones((K, C, 7, 7), device=DEV)
    gp = torch.ones((prois.shape[0], feats_np[0].shape[1], 7, 7), device=DEV)

    def runs():
        f = feat.detach().requires_grad_(True)
        p = [x.detach().requires_grad_(True) for x in pyr]
        return {
            "pool": lambda: modules.RoIPool((7, 7), 1.0)(f, rois5).backward(go),
            "msalign": lambda: modules.MultiScaleRoIAlign(["0", "1", "2", "3"], 7, 2)(
                {str(i): x for i, x in enumerate(p)}, dev(prois), [(256, 320)] * 2).backward(gp),
            "align_op": lambda: torch.ops.frr.roi_align(f, rois5, 1.0, 7, 7, 2, False).backward(go),
        }

    prev = torch.are_deterministic_algorithms_enabled()
    try:
        torch.use_deterministic_algorithms(True)
        for name, fn in runs().items():
            assert backward_kernels(fn) == ["roi_bwd_det_kernel"], name
        torch.use_deterministic_algorithms(False)
        want = {"pool": VARIANT_KERNELS[ops.roi_variant("roi_pool_bwd", K, B, C, fh, fw)["kernel"]],
                "align_op": VARIANT_KERNELS[ops.roi_variant("roi_align_bwd", K, B, C, fh, fw)["kernel"]]}
        want["msalign"] = sorted({k for f in feats_np for k in VARIANT_KERNELS[
            ops.roi_variant("roi_align_bwd", prois.shape[0], 2, f.shape[1], f.shape[2], f.shape[3])["kernel"]]})
        for name, fn in runs().items():
            assert backward_kernels(fn) == sorted(want[name]), name
    finally:
        torch.use_deterministic_algorithms(prev)


def test_opcheck_with_the_flag_on(det_flag):
    from faster_rcnn_pytorch_b200 import torch_ops  # noqa: F401
    B, C, fh, fw, K = 2, 16, 20, 30, 40
    feat = dev(synth.features(990, B, C, fh, fw))
    rois5 = dev(synth.random_rois(991, K, fh, fw, B))
    _, arg = ops.roi_pool_forward(feat, rois5)
    go = dev(grad_out(992, K, C))
    for op, args in ((torch.ops.frr._roi_pool_backward, (go, rois5, arg, 1.0, 7, 7, B, C, fh, fw)),
                     (torch.ops.frr._roi_align_backward, (go, rois5, 0.5, 7, 7, B, C, fh, fw, 2, False))):
        torch.library.opcheck(op, args, test_utils=("test_schema", "test_faketensor"))
    want = ops.roi_align_backward(go, rois5, (B, C, fh, fw), 0.5, 2, deterministic=True)
    assert torch.equal(torch.ops.frr._roi_align_backward(go, rois5, 0.5, 7, 7, B, C, fh, fw, 2, False), want)
