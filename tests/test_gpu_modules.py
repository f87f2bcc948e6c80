"""GPU parity of the drop-in call sites (faster_rcnn_pytorch_b200.modules / .anchor): same names, arguments and
return types as models/model.py:6-9,288-298 and anchor.py:7-55 -- these tests read like the reference's
own forward pass, one image per call."""
import numpy as np
import pytest
import torch

from conftest import golden
from faster_rcnn_pytorch_b200 import modules, ops, synth
from faster_rcnn_pytorch_b200.anchor import FRCNNAnchorMaker

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL = 1e-5


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def test_anchor_maker_drop_in(oracle):
    g = golden("anchors")
    am = FRCNNAnchorMaker()
    assert np.array_equal(am.anchor_base, g["base"])
    a = am._enumerate_shifted_anchor((64, 96))               # host numpy, like the reference
    assert isinstance(a, np.ndarray) and a.dtype == np.float32 and np.array_equal(a, g["full_64x96"])
    d = am.anchors_on(DEV, (600, 1000))
    assert d.is_cuda and d.shape == (20646, 4) and am.anchors_on(DEV, (600, 1000)) is d      # cached per size
    assert np.array_equal(d[:27].cpu().numpy(), g["head_600x1000"])
    am2 = FRCNNAnchorMaker(ratios=[1, 2], anchor_scales=[4, 8, 16])                          # non-default table
    want = oracle.enumerate_anchors((64, 96), table=am2.anchor_base)
    assert np.array_equal(am2._enumerate_shifted_anchor((64, 96)), want)


@pytest.mark.parametrize("key", ["rand_102_1000_0.7", "rand_103_3000_0.3", "rand_104_12000_0.7", "rand_106_300_0.3",
                                 "rand_107_1_0.7", "ties_110_500_0.5"])
def test_nms_drop_in_unsorted_input(oracle, key):
    """torchvision.ops.nms signature: unsorted boxes + scores -> int64 indices by decreasing score."""
    g = golden("nms")
    kind, seed, n, thr = key.split("_")
    b, s = synth.random_boxes(int(seed), int(n))
    if kind == "ties":
        s = (np.round(s * 8) / 8).astype(np.float32)
    keep = modules.nms(dev(b), dev(s), float(thr))
    assert keep.dtype == torch.int64 and keep.is_cuda
    assert np.array_equal(keep.cpu().numpy(), g[key].astype(np.int64))


def test_nms_drop_in_more_boxes_than_the_reference_path(oracle):
    """torchvision.ops.nms has no size limit: 20 000 boxes (beyond frr_topk_desc_opt's 16 384) still give the CPU kernel's list."""
    b, s = synth.random_boxes(123, 20000, cluster=False)
    b = (b * np.float32(0.2) + np.float32(0.4) * np.random.RandomState(3).uniform(size=(20000, 1)).astype(np.float32)).astype(np.float32)
    keep = modules.nms(dev(b), dev(s), 0.5)
    assert np.array_equal(keep.cpu().numpy(), oracle.nms(b, s, 0.5))


def test_nms_drop_in_edge_cases():
    e = modules.nms(torch.zeros((0, 4), device=DEV), torch.zeros((0,), device=DEV), 0.5)
    assert e.dtype == torch.int64 and e.numel() == 0
    with pytest.raises(RuntimeError):
        modules.nms(torch.zeros((3, 5), device=DEV), torch.zeros((3,), device=DEV), 0.5)
    with pytest.raises(ValueError, match="no CPU path"):
        modules.nms(torch.zeros((3, 4)), torch.zeros((3,)), 0.5)


@pytest.mark.parametrize("name,hw,seed,mode", [("small_train", (160, 256), 200, "train"), ("small_test", (160, 256), 201, "test"),
                                               ("voc_test", (600, 1000), 1000, "test"), ("rpn_train", (608, 1008), 2000, "train")])
def test_region_proposal_module(oracle, name, hw, seed, mode):
    """RegionProposal().forward(cls [N,2], reg [N,4], anchor [N,4], mode) -> ragged rois."""
    g = golden("proposal")
    logits, reg, _ = synth.rpn_head_outputs(seed, hw)
    anchor = FRCNNAnchorMaker()._enumerate_shifted_anchor(hw)
    rp = modules.RegionProposal()
    rois = rp(dev(logits), dev(reg), torch.from_numpy(anchor).to(DEV), mode)
    assert rois.dim() == 2 and rois.shape[1] == 4 and not rois.requires_grad
    # stage-wise oracle on the GPU's own fp32 scores / boxes (softmax + exp differ CPU<->GPU by ulps)
    boxes, scores, valid = ops.rpn_decode(dev(reg[None]), dev(logits[None]), anchors=dev(anchor))
    want = oracle.region_proposal(logits, reg, anchor, mode, scores=scores[0].cpu().numpy())
    if np.array_equal(want["boxes"], boxes[0].cpu().numpy()):
        assert np.array_equal(rois.cpu().numpy(), want["rois"])
    else:
        bx, va, sc = boxes[0].cpu().numpy(), valid[0].cpu().numpy().astype(bool), scores[0].cpu().numpy()
        pre_k, post_k = oracle.PROPOSAL_MODES[mode]
        src = np.nonzero(va)[0]
        order = oracle.sort_desc(sc[va])[:pre_k]
        tb = bx[src[order]]
        keep = oracle.nms(tb, -np.arange(len(tb), dtype=np.float32), 0.7)[:post_k]
        assert np.array_equal(rois.cpu().numpy(), tb[keep])
    # against the reference's own output: same number of rois and the same boxes up to exp() ulps, unless a
    # borderline pair flipped (then the count differs and only the stage-wise check above applies)
    # (a flip removes / inserts one roi and shifts the rows after it, so rows are compared as a set, not by position)
    assert abs(rois.shape[0] - int(g[f"{name}_nrois"])) <= 2
    head = g[f"{name}_rois_head"]
    got = rois.cpu().numpy()
    matched = [bool(np.isclose(got, h[None], rtol=1e-4, atol=1e-6).all(axis=1).any()) for h in head]
    assert np.mean(matched) >= 0.98, f"only {np.mean(matched):.3f} of the reference's first rois are among the GPU rois"


def test_target_maker_modules_like_the_reference_forward(oracle):
    """models/model.py:324-328 call pattern with torch.manual_seed controlling the sampling."""
    g = golden("targets")
    hw = (600, 1000)
    gt = np.array([[0.1, 0.2, 0.5, 0.7], [0.3, 0.3, 0.9, 0.95]], np.float32)
    lab = np.array([11, 14], np.int64)
    anchor = torch.from_numpy(FRCNNAnchorMaker()._enumerate_shifted_anchor(hw)).to(DEV)
    torch.manual_seed(7)
    cls_t, reg_t = modules.RPNTargetMaker()(dev(gt), anchor)
    assert cls_t.shape == (20646,) and cls_t.dtype == torch.int64 and reg_t.shape == (20646, 4)
    assert np.array_equal(cls_t.cpu().numpy(), g["kat6_rpn_cls"].astype(np.int64))
    rois, _ = synth.random_boxes(7 + 50, 2000)
    torch.manual_seed(8)
    fc, fr, fs = modules.FastRcnnTargetMaker()([dev(gt)], [dev(lab)], dev(rois))
    assert fc.shape == (128,) and fr.shape == (128, 4) and fs.shape == (128, 4)
    assert np.array_equal(fc.cpu().numpy(), g["kat6_frcnn_cls"].astype(np.int64))
    assert np.array_equal(fs.cpu().numpy(), g["kat6_frcnn_rois"])
    np.testing.assert_allclose(fr.cpu().numpy(), g["kat6_frcnn_reg"], rtol=RTOL, atol=2e-5)
    # float labels are accepted like models/model.py:416 (cast at :166)
    torch.manual_seed(8)
    fc2, _, _ = modules.FastRcnnTargetMaker()([dev(gt)], [dev(lab.astype(np.float32))], dev(rois))
    assert torch.equal(fc, fc2)


def test_roi_pool_module_in_a_head_forward_backward(oracle):
    """FastRCNNHead.forward (models/model.py:104-119): scale rois, RoIPool((7,7),1.0), view, Linear; backward
    reaches the feature map through the custom autograd function."""
    feat = dev(synth.features(800, 1, 32, 37, 62)).requires_grad_(True)
    b, _ = synth.random_boxes(801, 128)
    rois = dev(b) * torch.tensor([62, 37, 62, 37], dtype=torch.float32, device=DEV)
    pool = modules.RoIPool(output_size=(7, 7), spatial_scale=1.)
    x = pool(feat, [rois])
    assert x.shape == (128, 32, 7, 7) and x.is_contiguous()
    lin = torch.nn.Linear(32 * 49, 5).to(DEV)
    lin(x.view(x.size(0), -1)).sum().backward()
    wo, wa = oracle.roi_pool_forward(feat.detach().cpu().numpy(), oracle.scale_rois(b, 37, 62))
    assert np.array_equal(x.detach().cpu().numpy(), wo)
    go = lin.weight.detach().sum(0).reshape(1, 32, 7, 7).expand(128, -1, -1, -1).contiguous().cpu().numpy()
    want = oracle.roi_pool_backward(go, wa, oracle.scale_rois(b, 37, 62), (1, 32, 37, 62))
    scale = np.abs(want).max()
    assert np.abs(feat.grad.cpu().numpy() - want).max() <= 1e-5 * scale


def test_fpn_variant_target_maker_modules(oracle):
    """models/new_model.py call pattern: RPNTargetMaker()(boxes, anchors), FRCNNTargetMaker()(boxes, labels, rois)."""
    g = golden("targets_fpn")
    hw = (320, 480)
    anchors = dev(oracle.enumerate_anchors(hw))
    gt, lab = synth.gt_boxes(7000, 5)
    torch.manual_seed(7000)
    label, tg = modules.fpn.RPNTargetMaker()(dev(gt), anchors)
    assert label.dtype == torch.int64 and np.array_equal(label.cpu().numpy(), g["a_rpn_cls"].astype(np.int64))
    rois, _ = synth.random_boxes(7050, 2000)
    torch.manual_seed(7001)
    fc, fr, fs = modules.fpn.FRCNNTargetMaker()(dev(gt), dev(lab + 1), dev(rois))
    assert fc.shape == (512,) and np.array_equal(fc.cpu().numpy(), g["a_frcnn_cls"].astype(np.int64))
    assert np.array_equal(fs.cpu().numpy(), g["a_frcnn_rois"])


def test_multiscale_roi_align_module_matches_torchvision_call():
    """modules.MultiScaleRoIAlign(['0','1','2','3'], 7, 2)(features, [boxes], [image_shape]) -- models/new_model.py:127,143."""
    from conftest import golden
    from faster_rcnn_pytorch_b200 import modules
    g = golden("msroialign")
    feats_np, rois5 = synth.pyramid_inputs(image_hw=(256, 320))
    B = feats_np[0].shape[0]
    x = {str(i): torch.from_numpy(f).to("cuda:0") for i, f in enumerate(feats_np)}
    x["pool"] = torch.zeros(1, device="cuda:0")                     # extra map the pooler must ignore (featmap_names)
    order = np.concatenate([np.nonzero(rois5[:, 0] == b)[0] for b in range(B)])
    boxes = [torch.from_numpy(rois5[rois5[:, 0] == b, 1:]).to("cuda:0") for b in range(B)]
    pool = modules.MultiScaleRoIAlign(["0", "1", "2", "3"], 7, 2)
    out = pool(x, boxes, [(320, 256)] * B)                          # the reference passes (w, h)
    np.testing.assert_allclose(out.cpu().numpy(), g["wh_like_reference_out"][order], rtol=1e-5, atol=1e-6)


def test_joint_training_step_through_autograd():
    """A reference-shaped VGG16 Faster R-CNN (tools/frcnn_harness.py) takes two SGD steps with every region-stage op from
    libfrr: proposals -> device-sampled targets -> RoIPool (autograd) -> fused loss.  Gradients must reach the backbone
    through both the RoIPool backward kernel and the loss kernel's RPN gradients, and be finite."""
    import os, sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import frcnn_harness as fh
    from faster_rcnn_pytorch_b200 import targets
    torch.manual_seed(0)
    model = fh.FRCNNTrain(21, width_div=16).to("cuda:0").to(memory_format=torch.channels_last)
    opt = torch.optim.SGD(model.parameters(), lr=1e-3)
    gen = targets.DeviceGenerator("cuda:0")
    x, gt, lab = fh.make_batch(2, (160, 256), 3, "cuda:0", seed=1)
    first = model.extractor[0].weight.detach().clone()
    losses = []
    for _ in range(2):
        opt.zero_grad(set_to_none=True)
        loss = model(x, gt, lab, gen)
        assert loss.shape == (2, 5) and bool(torch.isfinite(loss).all())
        loss[:, 0].mean().backward()
        for name, p in model.named_parameters():
            assert p.grad is not None and bool(torch.isfinite(p.grad).all()), name
        opt.step()
        losses.append(loss.detach().cpu().numpy())
    assert float(model.extractor[0].weight.grad.abs().sum()) > 0           # the backbone received gradients
    assert float(model.reg_head.weight.grad.abs().sum()) > 0               # through the in-kernel class-row gather
    assert not torch.equal(first, model.extractor[0].weight.detach())
    np.testing.assert_allclose(losses[0][:, 0], losses[0][:, 1:].sum(axis=1), rtol=1e-5)


def test_torch_library_ops_match_the_module_path_and_pass_opcheck():
    """torch.ops.frr.{nms, roi_pool, roi_align, rpn_proposals}: same results as the Python wrappers, gradients through
    the registered autograd formulas, and torch.library.opcheck (schema, fake kernel, autograd registration)."""
    from faster_rcnn_pytorch_b200 import region, torch_ops  # noqa: F401
    feat = dev(synth.features(610, 2, 16, 20, 30)).requires_grad_(True)
    rois5 = dev(synth.random_rois(611, 40, 20, 30, 2))
    out, arg = torch.ops.frr.roi_pool(feat, rois5, 1.0, 7, 7)
    want, warg = ops.roi_pool_forward(feat.detach(), rois5)
    assert torch.equal(out, want) and torch.equal(arg, warg)
    go = torch.randn_like(out)
    out.backward(go)
    # (rois thinner than 6 pixels are added with global atomics: same sums, fp32 order not fixed)
    ref = ops.roi_pool_backward(go, warg, rois5, feat.shape)
    assert float((feat.grad - ref).abs().max()) <= 1e-5 * float(ref.abs().max())
    f2 = feat.detach().clone().requires_grad_(True)
    oa = torch.ops.frr.roi_align(f2, rois5, 0.5, 7, 7, 2, False)
    assert torch.equal(oa, ops.roi_align_forward(f2.detach(), rois5, spatial_scale=0.5, sampling_ratio=2))
    oa.backward(go)
    assert torch.equal(f2.grad, ops.roi_align_backward(go, rois5, f2.shape, spatial_scale=0.5, sampling_ratio=2))
    b, s = synth.random_boxes(612, 700)
    assert torch.equal(torch.ops.frr.nms(dev(b), dev(s), 0.5), modules.nms(dev(b), dev(s), 0.5))
    hw = (160, 256)
    _, reg, sc = synth.rpn_head_outputs(613, hw)
    r1, c1 = torch.ops.frr.rpn_proposals(dev(sc[None]), dev(reg[None]), hw[0], hw[1], 12000, 2000, 0.7, float(np.float32(0.001)))
    r2, c2 = region.rpn_proposals(dev(sc[None]), dev(reg[None]), image_hw=hw, mode="train")
    assert torch.equal(r1, r2) and torch.equal(c1, c2)
    for op, args in ((torch.ops.frr.roi_pool, (feat.detach().requires_grad_(True), rois5, 1.0, 7, 7)),
                     (torch.ops.frr.roi_align, (feat.detach().requires_grad_(True), rois5, 1.0, 7, 7, 2, False))):
        torch.library.opcheck(op, args, test_utils=("test_schema", "test_faketensor", "test_autograd_registration"))
