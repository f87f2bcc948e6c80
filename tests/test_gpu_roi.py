"""GPU parity: RoIPool / RoIAlign forward + backward (C ABI) vs the CPU oracle and the torchvision-CPU goldens.
RoIPool max + argmax bit-exact; backward and RoIAlign within 1e-5 relative (north_star)."""
import numpy as np
import pytest
import torch

from conftest import golden, sha
from faster_rcnn_pytorch_b200 import ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL, ATOL = 1e-5, 1e-6


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def close_accum(got, want):
    """Gradients are sums of many signed terms accumulated in a different fp32 order than the CPU loop:
    1e-5 relative is taken against the scale of the tensor (max |want|), the usual norm-wise bound."""
    scale = max(float(np.abs(want).max()), 1e-30)
    assert float(np.abs(got - want).max()) <= 1e-5 * scale


CASES = [("a", 500, 1, 8, 37, 62, 64), ("b", 501, 2, 16, 10, 14, 40), ("c", 502, 1, 4, 5, 6, 30)]


@pytest.mark.parametrize("name,seed,B,C,fh,fw,K", CASES)
@pytest.mark.parametrize("channels_last", [False, True])
def test_roi_pool_goldens(name, seed, B, C, fh, fw, K, channels_last):
    g = golden("roi")
    feat = dev(synth.features(seed, B, C, fh, fw))
    if channels_last:
        feat = feat.contiguous(memory_format=torch.channels_last)
    rois5 = dev(synth.random_rois(seed + 1, K, fh, fw, B))
    go = dev(np.random.RandomState(seed + 2).standard_normal((K, C, 7, 7)).astype(np.float32))
    out, arg = ops.roi_pool_forward(feat, rois5)
    assert np.array_equal(out.cpu().numpy(), g[f"{name}_pool_out"])          # bit-exact max
    assert np.array_equal(arg.cpu().numpy(), g[f"{name}_pool_argmax"])       # bit-exact argmax
    gin = ops.roi_pool_backward(go, arg, rois5, feat.shape, channels_last=channels_last)
    assert gin.is_contiguous(memory_format=torch.channels_last if channels_last else torch.contiguous_format)
    close_accum(gin.cpu().numpy(), g[f"{name}_pool_gin"])


@pytest.mark.parametrize("name,seed,B,C,fh,fw,K", CASES)
@pytest.mark.parametrize("scale", [1.0, 0.5])
@pytest.mark.parametrize("channels_last", [False, True])
def test_roi_align_goldens(name, seed, B, C, fh, fw, K, scale, channels_last):
    g = golden("roi")
    feat = dev(synth.features(seed, B, C, fh, fw))
    if channels_last:
        feat = feat.contiguous(memory_format=torch.channels_last)
    rois5 = dev(synth.random_rois(seed + 1, K, fh, fw, B))
    go = dev(np.random.RandomState(seed + 2).standard_normal((K, C, 7, 7)).astype(np.float32))
    out = ops.roi_align_forward(feat, rois5, spatial_scale=scale, sampling_ratio=2, aligned=False)
    np.testing.assert_allclose(out.cpu().numpy(), g[f"{name}_align_out_{scale}"], rtol=RTOL, atol=ATOL)
    gin = ops.roi_align_backward(go, rois5, feat.shape, spatial_scale=scale, sampling_ratio=2, aligned=False,
                                 channels_last=channels_last)
    close_accum(gin.cpu().numpy(), g[f"{name}_align_gin_{scale}"])


def test_head_call_path_list_of_rois(oracle):
    """models/model.py:104-113: roi * [fw,fh,fw,fh], list-of-tensors input, RoIPool((7,7), 1.0)."""
    g = golden("roi")
    feat = dev(synth.features(510, 1, 8, 37, 62))
    b, _ = synth.random_boxes(511, 32)
    scaled = dev(b) * torch.tensor([62, 37, 62, 37], dtype=torch.float32, device=DEV)
    out = ops.roi_pool(feat, [scaled], (7, 7), 1.0)
    assert np.array_equal(out.cpu().numpy(), g["head_pool_out"])


@pytest.mark.parametrize("B,C,fh,fw,K", [(2, 512, 37, 62, 256), (1, 512, 50, 83, 300), (3, 24, 37, 62, 100)])
def test_roi_pool_full_size_vs_oracle(oracle, B, C, fh, fw, K):
    feat = synth.features(700, B, C, fh, fw)
    rois5 = synth.random_rois(701, K, fh, fw, B)
    go = np.random.RandomState(702).standard_normal((K, C, 7, 7)).astype(np.float32)
    want_out, want_arg = oracle.roi_pool_forward(feat, rois5)
    out, arg = ops.roi_pool_forward(dev(feat), dev(rois5))
    assert np.array_equal(out.cpu().numpy(), want_out)
    assert np.array_equal(arg.cpu().numpy(), want_arg)
    gin = ops.roi_pool_backward(dev(go), arg, dev(rois5), feat.shape)
    close_accum(gin.cpu().numpy(), oracle.roi_pool_backward(go, want_arg, rois5, feat.shape))
    out_na, arg_na = ops.roi_pool_forward(dev(feat), dev(rois5), want_argmax=False)
    assert arg_na is None and torch.equal(out_na, out)


LONG_ROI_SHAPE = (24, 37, 62)                                             # C, fh, fw
LONG_ROI_CASES = [(3000, 2, True), (6000, 3, True), (1500, 1, False)]     # K, B, want_argmax


@pytest.mark.parametrize("K,B,want_argmax", LONG_ROI_CASES)
def test_roi_pool_forward_long_roi_lists(K, B, want_argmax):
    """more rois than one scan round of the forward kernel holds (2688) and more rois of one image than one list round
    (448), images interleaved, a few masked rows -- max and argmax bit-equal to torchvision's RoIPool (sha256 of both
    arrays and their values at sampled positions, made with torchvision 0.26's CPU kernel by
    tests/golden/make_golden_roi_long.py)"""
    g = golden("roi_long")
    key = f"{K}_{B}"
    C, fh, fw = LONG_ROI_SHAPE
    feat = dev(synth.features(710, B, C, fh, fw))
    rois5 = _mixed_rois(711, K, fh, fw, B, small_frac=0.2)
    keep = rois5[:, 0] >= 0
    out, arg = ops.roi_pool_forward(feat, dev(rois5), want_argmax=want_argmax)
    k = torch.from_numpy(keep).to(DEV)
    got = {"out": out[k].cpu().numpy()}
    if want_argmax:
        got["argmax"] = arg[k].cpu().numpy()
    for name, a in got.items():
        assert a.shape == tuple(g[f"{key}_shape"]), name
        assert np.array_equal(a.reshape(-1)[g[f"{key}_idx"]], g[f"{key}_{name}_sample"]), name
        assert np.array_equal(sha(a), g[f"{key}_{name}_sha"]), name


@pytest.mark.parametrize("B,C,fh,fw,K,scale,sr,aligned", [(2, 256, 50, 84, 200, 1.0, 2, False), (1, 256, 25, 42, 100, 0.5, 2, True),
                                                          (1, 16, 30, 30, 50, 1.0, -1, False)])
def test_roi_align_full_size_vs_oracle(oracle, B, C, fh, fw, K, scale, sr, aligned):
    feat = synth.features(710, B, C, fh, fw)
    rois5 = synth.random_rois(711, K, int(fh / scale), int(fw / scale), B)
    go = np.random.RandomState(712).standard_normal((K, C, 7, 7)).astype(np.float32)
    out = ops.roi_align_forward(dev(feat), dev(rois5), spatial_scale=scale, sampling_ratio=sr, aligned=aligned)
    np.testing.assert_allclose(out.cpu().numpy(), oracle.roi_align_forward(feat, rois5, spatial_scale=scale, sampling_ratio=sr, aligned=aligned),
                               rtol=RTOL, atol=ATOL)
    gin = ops.roi_align_backward(dev(go), dev(rois5), feat.shape, spatial_scale=scale, sampling_ratio=sr, aligned=aligned)
    close_accum(gin.cpu().numpy(), oracle.roi_align_backward(go, rois5, feat.shape, spatial_scale=scale, sampling_ratio=sr, aligned=aligned))


def _mixed_rois(seed, K, fh, fw, B, small_frac=0.4):
    """random rois, a share of them thinner than 7 feature pixels (bin size < 1: coinciding windows), interleaved images,
    a few masked (-1) rows"""
    rs = np.random.RandomState(seed)
    rois5 = synth.random_rois(seed, K, fh, fw, B)
    small = rs.rand(K) < small_frac
    for k in np.nonzero(small)[0]:
        x1, y1 = rs.uniform(0, fw - 1), rs.uniform(0, fh - 1)
        w = rs.uniform(0.2, 6.0) if rs.rand() < 0.7 else rs.uniform(6.0, fw / 2)
        h = rs.uniform(0.2, 6.0) if rs.rand() < 0.7 else rs.uniform(6.0, fh / 2)
        rois5[k, 1:] = [x1, y1, min(x1 + w, fw - 0.01), min(y1 + h, fh - 0.01)]
    rois5[:, 0] = rs.randint(0, B, size=K)
    rois5[rs.rand(K) < 0.03, 0] = -1
    return rois5.astype(np.float32)


@pytest.mark.parametrize("B,C,fh,fw,K,relu,channels_last", [
    (2, 32, 37, 62, 300, False, False),     # 8 planes per CTA, two CTAs per SM
    (2, 20, 37, 62, 200, True, False),      # partial last channel group (20 = 8 + 8 + 4), post-ReLU ties at 0
    (1, 16, 30, 40, 1300, True, False),     # > 512 rois of one image: several list rounds
    (1, 16, 50, 83, 700, True, False),      # 800x1333 map: every roi through the streaming atomic kernel
    (2, 12, 50, 83, 300, False, True),      # ... with a channels_last gradient
    (3, 16, 37, 62, 400, True, True),       # channels_last gradient
    (1, 8, 110, 110, 150, False, False),    # 48 KB planes
    (2, 7, 20, 20, 100, True, False),       # partial single channel group, odd channel count (a warp with one plane)
])
def test_roi_pool_backward_colour_kernel(oracle, B, C, fh, fw, K, relu, channels_last):
    """roi_pool_bwd_color_kernel (colour classes, rois of >= 6 pixels per side) + roi_pool_bwd_tail_kernel (the smaller
    rois, global atomics) against the CPU loop, on the forward's own argmax."""
    feat = synth.features(740, B, C, fh, fw)
    if relu:
        feat = np.maximum(feat, 0.0)  # VGG features are post-ReLU: whole windows of zeros, argmax ties
    rois5 = _mixed_rois(741, K, fh, fw, B)
    go = np.random.RandomState(742).standard_normal((K, C, 7, 7)).astype(np.float32)
    f = dev(feat)
    if channels_last:
        f = f.contiguous(memory_format=torch.channels_last)
    out, arg = ops.roi_pool_forward(f, dev(rois5))
    live = rois5[:, 0] >= 0
    wo, wa = oracle.roi_pool_forward(feat, rois5[live])
    assert np.array_equal(out.cpu().numpy()[live], wo) and np.array_equal(arg.cpu().numpy()[live], wa)
    gin = ops.roi_pool_backward(dev(go), arg, dev(rois5), feat.shape, channels_last=channels_last)
    want = oracle.roi_pool_backward(go[live], wa, rois5[live], feat.shape)
    close_accum(gin.cpu().numpy(), want)
    if fh * fw > 2300:
        return  # maps above 37 x 62 take the streaming atomic kernel for every roi (fp32 order not fixed)
    # rois of at least 6 x 6 pixels never leave the shared-memory path: fixed summation order, bit-reproducible
    big = synth.random_rois(743, K, fh, fw, B)
    big[:, 3] = np.maximum(big[:, 3], big[:, 1] + 7.0)
    big[:, 4] = np.maximum(big[:, 4], big[:, 2] + 7.0)
    _, arg_b = ops.roi_pool_forward(f, dev(big))
    g1 = ops.roi_pool_backward(dev(go), arg_b, dev(big), feat.shape, channels_last=channels_last)
    g2 = ops.roi_pool_backward(dev(go), arg_b, dev(big), feat.shape, channels_last=channels_last)
    assert torch.equal(g1, g2)


@pytest.mark.parametrize("channels_last", [False, True])
def test_roi_align_backward_stream_kernel(oracle, channels_last):
    """50x84 map: the separable plane kernel would be left with 8 planes per SM, roi_align_bwd_stream_kernel (one CTA per
    roi, merged taps in registers, global atomics) runs instead -- both memory formats, rois crossing the borders."""
    B, C, fh, fw, K = 2, 40, 50, 84, 150
    rois5 = synth.random_rois(751, K, fh, fw, B)
    rois5[0, 1:] = [-30, -30, -20, -20]          # entirely outside: contributes nothing
    rois5[1, 1:] = [10.2, 10.2, 10.6, 10.5]      # sub-pixel roi: all samples of a bin on the same pixels (merged taps)
    go = np.random.RandomState(752).standard_normal((K, C, 7, 7)).astype(np.float32)
    gin = ops.roi_align_backward(dev(go), dev(rois5), (B, C, fh, fw), spatial_scale=1.0, sampling_ratio=2, aligned=False,
                                 channels_last=channels_last)
    assert gin.is_contiguous(memory_format=torch.channels_last if channels_last else torch.contiguous_format)
    close_accum(gin.cpu().numpy(), oracle.roi_align_backward(go, rois5, (B, C, fh, fw), spatial_scale=1.0, sampling_ratio=2,
                                                             aligned=False))


def test_large_planes_take_the_direct_kernels(oracle):
    """FPN level-0 sized map (200x336 = 262 KB per plane) does not fit shared memory."""
    B, C, fh, fw, K = 1, 4, 200, 336, 60
    feat = synth.features(720, B, C, fh, fw)
    rois5 = synth.random_rois(721, K, fh, fw, B)
    go = np.random.RandomState(722).standard_normal((K, C, 7, 7)).astype(np.float32)
    out, arg = ops.roi_pool_forward(dev(feat), dev(rois5))
    wo, wa = oracle.roi_pool_forward(feat, rois5)
    assert np.array_equal(out.cpu().numpy(), wo) and np.array_equal(arg.cpu().numpy(), wa)
    gin = ops.roi_pool_backward(dev(go), arg, dev(rois5), feat.shape)
    close_accum(gin.cpu().numpy(), oracle.roi_pool_backward(go, wa, rois5, feat.shape))
    oa = ops.roi_align_forward(dev(feat), dev(rois5), spatial_scale=1.0, sampling_ratio=2)
    np.testing.assert_allclose(oa.cpu().numpy(), oracle.roi_align_forward(feat, rois5), rtol=RTOL, atol=ATOL)
    ga = ops.roi_align_backward(dev(go), dev(rois5), feat.shape)
    close_accum(ga.cpu().numpy(), oracle.roi_align_backward(go, rois5, feat.shape))


def test_autograd_and_edge_cases(oracle):
    feat = dev(synth.features(730, 2, 12, 9, 11)).requires_grad_(True)
    rois5 = synth.random_rois(731, 20, 9, 11, 2)
    rois5[0, 1:] = [-50, -50, -40, -40]      # entirely outside: empty bins -> 0 / argmax -1
    rois5[1, 1:] = [3.2, 3.2, 3.3, 3.3]      # sub-pixel roi
    out = ops.roi_pool(feat, dev(rois5), 7, 1.0)
    wo, wa = oracle.roi_pool_forward(feat.detach().cpu().numpy(), rois5)
    assert np.array_equal(out.detach().cpu().numpy(), wo)
    go = torch.randn_like(out)
    out.backward(go)
    close_accum(feat.grad.cpu().numpy(), oracle.roi_pool_backward(go.cpu().numpy(), wa, rois5, tuple(feat.shape)))
    feat2 = feat.detach().clone().requires_grad_(True)
    oa = ops.roi_align(feat2, dev(rois5), 7, 1.0, sampling_ratio=2)
    oa.backward(go)
    close_accum(feat2.grad.cpu().numpy(), oracle.roi_align_backward(go.cpu().numpy(), rois5, tuple(feat.shape)))
    empty = ops.roi_pool(feat.detach(), torch.zeros((0, 5), device=DEV), 7, 1.0)
    assert empty.shape == (0, 12, 7, 7)
    with pytest.raises(ValueError):
        ops.roi_pool(feat.detach().cpu(), torch.zeros((1, 5)), 7, 1.0)


@pytest.mark.parametrize("tag,shapes", [("hw", [(256, 320)] * 2), ("wh_like_reference", [(320, 256)] * 2)])
@pytest.mark.parametrize("channels_last", [False, True])
def test_multiscale_roi_align_goldens(tag, shapes, channels_last):
    """MultiScaleRoIAlign(['0'..'3'], 7, 2)(x, boxes, image_shapes) as called at models/new_model.py:127,143: levels
    bit-exact (incl. boxes exactly on a LevelMapper boundary), output within 1e-5, feature gradients norm-wise 1e-5."""
    g = golden("msroialign")
    feats_np, rois5 = synth.pyramid_inputs(image_hw=(256, 320))
    feats = [dev(f) for f in feats_np]
    if channels_last:
        feats = [f.contiguous(memory_format=torch.channels_last) for f in feats]
    feats = [f.requires_grad_(True) for f in feats]
    scales, k_min, k_max = ops.infer_scales(feats, shapes)
    assert np.array_equal(np.asarray(scales), g[f"{tag}_scales"])
    out, levels = ops.multiscale_roi_align({str(i): f for i, f in enumerate(feats)}, dev(rois5), shapes, 7, 2,
                                           return_levels=True)
    assert np.array_equal(levels.cpu().numpy(), g[f"{tag}_levels"])
    np.testing.assert_allclose(out.detach().cpu().numpy(), g[f"{tag}_out"], rtol=RTOL, atol=ATOL)
    out.backward(dev(g["grad_out"]))
    for i, f in enumerate(feats):
        close_accum(f.grad.cpu().numpy(), g[f"{tag}_gin{i}"])


def test_multiscale_roi_align_list_boxes_and_oracle(oracle):
    """Boxes as the reference passes them (list of [L,4] per image) on a larger pyramid; checked against the oracle."""
    feats_np, rois5 = synth.pyramid_inputs(seed=8200, B=3, C=16, image_hw=(384, 512), K=300)
    order = np.concatenate([np.nonzero(rois5[:, 0] == b)[0] for b in range(3)])
    boxes = [dev(rois5[rois5[:, 0] == b, 1:]) for b in range(3)]
    shapes = [(384, 512)] * 3
    out, levels = ops.multiscale_roi_align([dev(f) for f in feats_np], boxes, shapes, 7, 2, return_levels=True)
    want, lv = oracle.multiscale_roi_align(feats_np, rois5[order], shapes)
    assert np.array_equal(levels.cpu().numpy().astype(np.int64), lv)
    np.testing.assert_allclose(out.cpu().numpy(), want, rtol=RTOL, atol=ATOL)
