"""torch.ops.frr.* of the batched region stage without a GPU: schemas, fake (meta) outputs at the configs' shapes, and
whole predict / train steps traced by make_fx on fake CUDA tensors into graphs of frr.* and aten.* calls only."""
import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode
from torch.fx.experimental.proxy_tensor import make_fx

import region_steps
from faster_rcnn_pytorch_b200 import ops, synth, targets

frr = torch.ops.frr
NEW_OPS = ("rpn_proposals_sized", "rpn_proposals_anchored", "rois5", "roi_pool_sized", "_roi_pool_backward_sized",
           "make_targets", "rpn_targets", "frcnn_targets", "region_loss", "decode_classwise", "class_nms", "pack_detections",
           "multiscale_roi_align", "_multiscale_roi_align_backward")
MUTATING = {"make_targets", "rpn_targets", "frcnn_targets"}       # mt_state, and nothing else


@pytest.fixture
def fake():
    with FakeTensorMode() as mode:
        yield mode


def cuda(*shape, dtype=torch.float32, device="cuda"):
    return torch.empty(shape, dtype=dtype, device=device)


def shapes(ts):
    return [(tuple(t.shape), t.dtype) for t in ts]


def test_every_op_exists_and_declares_only_mt_state_mutated():
    for name in NEW_OPS:
        schema = getattr(frr, name).default._schema
        mutated = [a.name for a in schema.arguments if a.alias_info is not None and a.alias_info.is_write]
        assert mutated == (["mt_state"] if name in MUTATING else []), (name, str(schema))
        assert all(r.alias_info is None for r in schema.returns), str(schema)


def test_proposals_fake_shapes(fake):
    N = synth.num_anchors((608, 1008))                   # configs[1]: 38 x 63 cells
    assert N == 21546
    out = frr.rpn_proposals(cuda(2, N, 2), cuda(2, N, 4), 608, 1008, 12000, 2000, 0.7, 0.001)
    assert shapes(out) == [((2, 2000, 4), torch.float32), ((2,), torch.int32)]
    Ng = 50 * 50 * 9                                     # mixed-size batch padded to 800 x 800
    out = frr.rpn_proposals_sized(cuda(3, Ng, 2), cuda(3, Ng, 4), cuda(3, 2, dtype=torch.int32), 50, 50, 6000, 300, 0.7, 0.001)
    assert shapes(out) == [((3, 300, 4), torch.float32), ((3,), torch.int32)]
    Nf = sum((800 // s) * (800 // s) for s in (4, 8, 16, 32, 64)) * 3       # FPN: five levels, three anchors per cell
    out = frr.rpn_proposals_anchored(cuda(2, Nf, 2), cuda(2, Nf, 4), cuda(Nf, 4), 2000, 1000, 0.7, 0.01)
    assert shapes(out) == [((2, 1000, 4), torch.float32), ((2,), torch.int32)]


def test_infer_plan_fake_shapes(fake):
    """region.InferPlan at configs[0] (one 600 x 1000 image, 21 classes) and configs[3] (8 x 800 x 1333, 81 classes)."""
    for B, hw, NC in ((1, (600, 1000), 21), (8, (800, 1333), 81)):
        fh, fw = hw[0] // 16, hw[1] // 16
        R, C = 300, 512
        rois, cnt = cuda(B, R, 4), cuda(B, dtype=torch.int32)
        r5 = frr.rois5(rois, cnt, fh, fw, None, 16)
        assert shapes([r5]) == [((B * R, 5), torch.float32)]
        pooled, arg = frr.roi_pool(cuda(B, C, fh, fw), r5, 1.0, 7, 7)
        assert shapes([pooled, arg]) == [((B * R, C, 7, 7), torch.float32), ((B * R, C, 7, 7), torch.int32)]
        prob, boxes = frr.decode_classwise(cuda(B * R, NC), cuda(B * R, 4 * NC), rois.view(-1, 4), NC)
        assert shapes([prob, boxes]) == [((B * R, NC), torch.float32), ((B * R, 4 * NC), torch.float32)]
        det = frr.class_nms(prob.view(B, R, NC), boxes.view(B, R, 4 * NC), NC, 0.05, 0.3, cnt, None)
        cap = R * (NC - 1)
        assert shapes(det) == [((B, cap, 4), torch.float32), ((B, cap), torch.int32), ((B, cap), torch.float32),
                               ((B,), torch.int32)]
        assert shapes(frr.class_nms(prob.view(B, R, NC), boxes.view(B, R, 4 * NC), NC, 0.05, 0.3, None, 64))[0] == \
            ((B, 64, 4), torch.float32)
        for rank, pcm in (("class", 0), ("score", 0), ("score", 100)):
            out = frr.pack_detections(*det, 100, cuda(B, 2), True, rank, pcm)
            assert shapes(out) == [((B, 100, 6), torch.float32), ((B,), torch.int32)]
        with pytest.raises(ValueError):
            frr.pack_detections(*det, 100, None, False, "best", 0)


def test_train_plan_fake_shapes(fake):
    """region.TrainPlan at configs[2] (16 x 600 x 1000, G = 8), uniform and with per-image sizes."""
    B, hw, G, C = 16, (600, 1000), 8, 512
    fh, fw = hw[0] // 16, hw[1] // 16
    N, S = fh * fw * 9, targets.FRCNN_BATCH
    gt, lab, props, pcnt = cuda(B, G, 4), cuda(B, G, dtype=torch.int64), cuda(B, 2000, 4), cuda(B, dtype=torch.int32)
    state = cuda(626, dtype=torch.int32)
    want = [((B, N), torch.int64), ((B, N, 4), torch.float32), ((B, S), torch.int64), ((B, S, 4), torch.float32),
            ((B, S, 4), torch.float32), ((B, S), torch.int32), ((B,), torch.int32)]
    for image_hw in (None, cuda(B, 2, dtype=torch.int32)):
        t = frr.make_targets(gt, None, lab, props, pcnt, state, hw[0], hw[1], image_hw)
        assert shapes(t) == want
        r5 = frr.rois5(t[4], t[6], fh, fw, image_hw, 16)
        assert shapes([r5]) == [((B * S, 5), torch.float32)]
    feat = cuda(B, C, fh, fw)
    pooled, arg = frr.roi_pool_sized(feat, r5, image_hw, 1.0, 7, 7, 16)
    assert shapes([pooled, arg]) == [((B * S, C, 7, 7), torch.float32), ((B * S, C, 7, 7), torch.int32)]
    g = frr._roi_pool_backward_sized(pooled, r5, arg, image_hw, 1.0, 7, 7, B, C, fh, fw, 16)
    assert shapes([g]) == [((B, C, fh, fw), torch.float32)]
    assert shapes(frr.rpn_targets(gt, None, state, None, hw[0], hw[1], None, "vgg")) == want[:2]
    assert shapes(frr.frcnn_targets(props, pcnt, gt, None, lab, state, "vgg")) == want[2:]
    assert shapes(frr.frcnn_targets(props, pcnt, gt, None, lab, state, "fpn")) == \
        [((B, 512), torch.int64), ((B, 512, 4), torch.float32), ((B, 512, 4), torch.float32), ((B, 512), torch.int32),
         ((B,), torch.int32)]
    anchors = cuda(12345, 4)
    assert shapes(frr.rpn_targets(gt, None, state, anchors, 0, 0, None, "fpn")) == \
        [((B, 12345), torch.int64), ((B, 12345, 4), torch.float32)]


def test_region_loss_fake_shapes(fake):
    B, N, S, NC = 16, 20646, 128, 21
    rc, rr, rt, rtr = cuda(B, N, 2), cuda(B, N, 4), cuda(B, N, dtype=torch.int64), cuda(B, N, 4)
    fc, ft, ftr = cuda(B, S, NC), cuda(B, S, dtype=torch.int64), cuda(B, S, 4)
    for fr in (cuda(B, S, NC * 4), cuda(B, S, NC, 4), cuda(B, S, 4)):
        out = frr.region_loss(rc, rr, rt, rtr, fc, fr, ft, ftr)
        assert shapes(out) == [((B, 5), torch.float32), ((B, N, 2), torch.float32), ((B, N, 4), torch.float32),
                               ((B, S, NC), torch.float32), (tuple(fr.shape), torch.float32)]
    out = frr.region_loss(rc, rr, rt, rtr, None, None, None, None)
    assert shapes(out)[0] == ((B, 5), torch.float32) and out[3].numel() == 0 and out[4].numel() == 0


def test_multiscale_roi_align_fake_shapes_and_autograd(fake):
    """FPN: four pooled levels (strides 4..32) of an 800 x 1088 batch; the backward gives one gradient per level."""
    B, C, K = 2, 256, 1000
    feats = [cuda(B, C, 800 // s, 1088 // s, device="meta").requires_grad_(True) for s in (4, 8, 16, 32)]
    scales, k_min, k_max = ops.infer_scales(feats, [(800, 1088)])
    assert (k_min, k_max) == (2, 5)
    rois = cuda(K, 5, device="meta")
    out, levels, per = frr.multiscale_roi_align(feats, rois, 7, 7, 2, scales, k_min, k_max, 224.0, 4)
    assert shapes([out, levels, per]) == [((K, C, 7, 7), torch.float32), ((K,), torch.int32), ((4, K, 5), torch.float32)]

    def fwd_bwd(rois, *feats):
        out = frr.multiscale_roi_align(list(feats), rois, 7, 7, 2, scales, k_min, k_max, 224.0, 4)[0]
        return torch.autograd.grad(out.sum(), feats)

    gm = make_fx(fwd_bwd, tracing_mode="fake")(rois, *feats)
    assert _only_frr_and_aten(gm) == {"multiscale_roi_align", "_multiscale_roi_align_backward"}
    assert [tuple(g.shape) for g in gm(rois, *feats)] == [tuple(f.shape) for f in feats]


def _targets_of(gm):
    return {str(n.target) for n in gm.graph.nodes if n.op == "call_function"}


def _only_frr_and_aten(gm):
    import operator
    calls = _targets_of(gm)
    bad = [c for c in calls if not (c.startswith("frr.") or c.startswith("aten.") or c == str(operator.getitem))]
    assert not bad, bad
    return {c.split(".")[1] for c in calls if c.startswith("frr.")}


def test_make_fx_predict_step(fake):
    B, grid, NC, C = 2, (50, 50), 21, 64
    N = grid[0] * grid[1] * 9
    args = (cuda(B, C, *grid), cuda(B, N, 2), cuda(B, N, 4), cuda(B, 2, dtype=torch.int32), cuda(C * 49, NC),
            cuda(C * 49, 4 * NC))
    gm = make_fx(lambda *a: region_steps.predict(*a, grid=grid, NC=NC), tracing_mode="fake")(*args)
    assert _only_frr_and_aten(gm) == {"rpn_proposals_sized", "rois5", "roi_pool_sized", "decode_classwise", "class_nms",
                                      "pack_detections"}
    packed, pc, rois, cnt = gm(*args)
    assert shapes([packed, pc]) == [((B, 100, 6), torch.float32), ((B,), torch.int32)]


@pytest.mark.parametrize("sized", [False, True])
def test_make_fx_train_step(fake, sized):
    B, hw, NC, C, G = 2, (320, 480), 21, 16, 5
    fh, fw = hw[0] // 16, hw[1] // 16
    N = fh * fw * 9

    def inputs(device):
        t = lambda *shape, dtype=torch.float32: cuda(*shape, dtype=dtype, device=device)      # noqa: E731
        return (t(B, C, fh, fw).requires_grad_(True), t(B, N, 2).requires_grad_(True), t(B, N, 4).requires_grad_(True),
                t(B, G, 4), t(B, dtype=torch.int32), t(B, G, dtype=torch.int64), t(B, 2000, 4), t(B, dtype=torch.int32),
                t(626, dtype=torch.int32), t(B, 2, dtype=torch.int32) if sized else None, t(C * 49, NC),
                t(C * 49, 4 * NC))

    fwd = make_fx(lambda *a: region_steps.train(*a, padded_hw=hw, NC=NC)[0], tracing_mode="fake")(*inputs("cuda"))
    pool = ("roi_pool_sized",) if sized else ("roi_pool",)
    assert _only_frr_and_aten(fwd) == {"make_targets", "rois5", "region_loss", *pool}
    args = inputs("meta")
    gm = make_fx(lambda *a: region_steps.train_grads(*a, padded_hw=hw, NC=NC), tracing_mode="fake")(*args)
    pool += ("_roi_pool_backward_sized",) if sized else ("_roi_pool_backward",)
    assert _only_frr_and_aten(gm) == {"make_targets", "rois5", "region_loss", *pool}
    loss, g_feat, g_cls, g_reg = gm(*args)
    assert shapes([loss, g_feat, g_cls, g_reg]) == [((B, 5), torch.float32), ((B, C, fh, fw), torch.float32),
                                                     ((B, N, 2), torch.float32), ((B, N, 4), torch.float32)]


def test_cpu_tensors_raise():
    cpu = torch.zeros
    with pytest.raises((NotImplementedError, RuntimeError)):
        frr.rois5(cpu((1, 4, 4)), None, 10, 10, None, 16)
    with pytest.raises((NotImplementedError, RuntimeError)):
        frr.rpn_proposals_sized(cpu((1, 90, 2)), cpu((1, 90, 4)), torch.zeros((1, 2), dtype=torch.int32), 10, 1, 100, 10,
                                0.7, 0.001)
    with pytest.raises((NotImplementedError, RuntimeError)):
        frr.decode_classwise(cpu((3, 2)), cpu((3, 8)), cpu((3, 4)), 2)
    with pytest.raises((NotImplementedError, RuntimeError)):
        frr.make_targets(cpu((1, 2, 4)), None, torch.zeros((1, 2), dtype=torch.int64), cpu((1, 3, 4)), None,
                         torch.zeros((626,), dtype=torch.int32), 64, 64, None)
    with pytest.raises((NotImplementedError, RuntimeError)):
        frr.multiscale_roi_align([cpu((1, 2, 8, 8)), cpu((1, 2, 4, 4))], cpu((3, 5)), 7, 7, 2, [0.25, 0.125], 2, 3, 224.0, 4)
