"""torch.ops.frr.* of the batched region stage on the device: every op equals the Python function it wraps bit for bit,
passes torch.library.opcheck, and whole predict / train steps compile with fullgraph=True (aot_eager, inductor, CUDA
graphs) to the results of the eager step while launching exactly its libfrr kernels."""
import contextlib

import numpy as np
import pytest
import torch

import region_steps
from faster_rcnn_pytorch_b200 import _lib, ops, region, synth, targets

pytestmark = pytest.mark.gpu

frr = torch.ops.frr
DEV = "cuda:0"
GRID = (20, 30)                                  # a 320 x 480 padded batch
PADDED = (GRID[0] * 16, GRID[1] * 16)
SIZES = [(320, 480), (240, 320), (300, 470)]
SIZES2 = [(320, 240), (200, 100), (320, 480)]
NC, C = 21, 16
OPCHECK = ("test_schema", "test_faketensor", "test_autograd_registration", "test_aot_dispatch_dynamic")


def hw_dev(sizes):
    return torch.tensor(sizes, dtype=torch.int32, device=DEV)


def rpn_head(B, seed, grid=GRID):
    g = torch.Generator().manual_seed(seed)
    N = grid[0] * grid[1] * 9
    return torch.randn((B, N, 2), generator=g).to(DEV), (torch.randn((B, N, 4), generator=g) * 0.2).to(DEV)


def feats(B, seed, grid=GRID):
    g = torch.Generator().manual_seed(seed)
    return torch.randn((B, C, *grid), generator=g).to(DEV)


def head_weights(seed):
    g = torch.Generator().manual_seed(seed)
    return ((torch.randn((C * 49, NC), generator=g) * 0.05).to(DEV),
            (torch.randn((C * 49, 4 * NC), generator=g) * 0.05).to(DEV))


def gt_batch(B, G, seed):
    rs = np.random.RandomState(seed)
    xy1 = rs.uniform(0.0, 0.7, (B, G, 2))
    wh = rs.uniform(0.05, 0.3, (B, G, 2))
    gt = torch.from_numpy(np.concatenate([xy1, xy1 + wh], axis=2).astype(np.float32)).to(DEV)
    count = torch.from_numpy(rs.randint(1, G + 1, B).astype(np.int32)).to(DEV)
    labels = torch.from_numpy(rs.randint(0, 20, (B, G)).astype(np.int64)).to(DEV)
    return gt, count, labels


def state(seed):
    torch.manual_seed(seed)
    return targets.DeviceGenerator(DEV)


def live(r5):
    return r5[:, 0] >= 0          # the RoI kernels leave the output rows of masked rois (batch index -1) unwritten


def equal(a, b):
    if isinstance(a, (tuple, list)):
        return len(a) == len(b) and all(equal(x, y) for x, y in zip(a, b))
    return torch.equal(a, b)


@contextlib.contextmanager
def deterministic(on=True):
    # warn_only: the head's cuBLAS matmuls have no deterministic-mode switch; the flag is read by the RoI backward ops
    prev = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(on, warn_only=True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev[0], warn_only=prev[1])


# ------------------------------------------------------------------------------------------------
# each op against the function it wraps
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["train", "test"])
def test_proposals_sized_and_anchored(mode):
    pre, post = region.PROPOSAL_MODES[mode]
    cls, reg = rpn_head(len(SIZES), 10)
    hw = hw_dev(SIZES)
    got = frr.rpn_proposals_sized(cls, reg, hw, *GRID, pre, post, 0.7, ops._MIN_SIZE)
    assert equal(got, region.rpn_proposals(cls, reg, image_hw=hw, grid_hw=GRID, mode=mode))
    fhws = [(PADDED[0] // s, PADDED[1] // s) for s in (4, 8, 16, 32, 64)]        # FPN: five levels
    anchors = ops.anchors_pyramid(fhws, PADDED, DEV)
    g = torch.Generator().manual_seed(11)
    fc = torch.randn((2, anchors.shape[0], 2), generator=g).to(DEV)
    fr = (torch.randn((2, anchors.shape[0], 4), generator=g) * 0.2).to(DEV)
    got = frr.rpn_proposals_anchored(fc, fr, anchors, pre, post, 0.7, 0.01)
    assert equal(got, region.rpn_proposals(fc, fr, anchors=anchors, mode=mode, min_size=0.01))


def test_rois5_and_roi_pool_sized():
    B = len(SIZES)
    hw = hw_dev(SIZES)
    rois, cnt = region.rpn_proposals(*rpn_head(B, 20), image_hw=hw, grid_hw=GRID, mode="test")
    assert torch.equal(frr.rois5(rois, cnt, *GRID, None, 16), ops.rois5(rois, cnt, GRID))
    r5 = frr.rois5(rois, cnt, *GRID, hw, 16)
    assert torch.equal(r5, ops.rois5(rois, cnt, GRID, image_hw=hw))
    f = feats(B, 21).requires_grad_(True)
    out, arg = frr.roi_pool_sized(f, r5, hw, 1.0, 7, 7, 16)
    want, warg = ops.roi_pool_forward(f.detach(), r5, image_hw=hw)
    m = live(r5)
    assert torch.equal(out[m], want[m]) and torch.equal(arg[m], warg[m])
    go = torch.randn_like(out)
    with deterministic():
        g_det, = torch.autograd.grad(out, f, go, retain_graph=True)
        assert torch.equal(g_det, ops.roi_pool_backward(go, arg, r5, f.shape, image_hw=hw))
    g, = torch.autograd.grad(out, f, go)
    ref = ops.roi_pool_backward(go, arg, r5, f.shape, image_hw=hw)
    assert float((g - ref).abs().max()) <= 1e-5 * float(ref.abs().max())


@pytest.mark.parametrize("sized", [False, True])
def test_make_targets(sized):
    B = len(SIZES)
    hw = hw_dev(SIZES) if sized else None
    props, pcnt = region.rpn_proposals(*rpn_head(B, 30), image_hw=hw if sized else PADDED, grid_hw=GRID, mode="train")
    gt, gc, gl = gt_batch(B, 6, 31)
    g_op, g_ref = state(32), state(32)
    got = frr.make_targets(gt, gc, gl, props, pcnt, g_op.state, *PADDED, hw)
    want = targets.make_targets(gt, gc, gl, props, pcnt, image_hw=PADDED if hw is None else hw, generator=g_ref,
                                grid_hw=GRID)
    keys = ("rpn_cls", "rpn_reg", "frcnn_cls", "frcnn_reg", "sample_rois", "keep_index", "n_samples")
    assert equal(got, [want[k] for k in keys])
    assert torch.equal(g_op.state, g_ref.state) and not torch.equal(g_op.state, state(32).state)


@pytest.mark.parametrize("variant", ["vgg", "fpn"])
def test_rpn_and_frcnn_targets(variant):
    B = 2
    gt, gc, gl = gt_batch(B, 7, 40)
    if variant == "vgg":
        anchors, kw = None, dict(image_hw=PADDED)
    else:
        anchors = ops.anchors_pyramid([(PADDED[0] // s, PADDED[1] // s) for s in (4, 8, 16, 32, 64)], PADDED, DEV)
        kw = dict(anchors=anchors)
    g_op, g_ref = state(41), state(41)
    got = frr.rpn_targets(gt, gc, g_op.state, anchors, *PADDED, None, variant)
    assert equal(got, targets.rpn_targets(gt, gc, generator=g_ref, variant=variant, **kw))
    assert torch.equal(g_op.state, g_ref.state)
    props, pcnt = region.rpn_proposals(*rpn_head(B, 42), image_hw=PADDED, mode="train")
    got = frr.frcnn_targets(props, pcnt, gt, gc, gl, g_op.state, variant)
    assert equal(got, targets.frcnn_targets(props, pcnt, gt, gc, gl, variant=variant, generator=g_ref))
    assert torch.equal(g_op.state, g_ref.state)


@pytest.mark.parametrize("reg_rows", ["head", "gathered", "rpn_only", "frcnn_only"])
def test_region_loss(reg_rows):
    d = synth.loss_inputs(N=2000, S=64)
    B = 2
    t = {k: torch.from_numpy(np.stack([v] * B)).to(DEV) for k, v in d.items()}
    t["frc_reg"] = t["frc_reg"].reshape(B, 64, -1) if reg_rows != "gathered" else t["frc_reg"][:, :, 0]
    preds = [t[k].clone().requires_grad_(True) for k in ("rpn_cls", "rpn_reg", "frc_cls", "frc_reg")]
    if reg_rows == "rpn_only":
        preds[2:] = [None, None]
    if reg_rows == "frcnn_only":
        preds[:2] = [None, None]
    rpn = (preds[0], preds[1], t["rpn_tcls"], t["rpn_treg"]) if preds[0] is not None else (None,) * 4
    frc = (preds[2], preds[3], t["frc_tcls"], t["frc_treg"]) if preds[2] is not None else (None,) * 4
    out = frr.region_loss(*rpn, *frc)
    ref = [p.detach().clone().requires_grad_(True) if p is not None else None for p in preds]
    rrpn = (ref[0], ref[1]) + rpn[2:] if ref[0] is not None else rpn
    rfrc = (ref[2], ref[3]) + frc[2:] if ref[2] is not None else frc
    want = ops.region_loss(*rrpn, *rfrc)
    assert torch.equal(out[0], want)
    up = torch.randn((B, 5), device=DEV)
    have = [p for p in preds if p is not None]
    got_g = torch.autograd.grad(out[0], have, up)
    want_g = torch.autograd.grad(want, [p for p in ref if p is not None], up, retain_graph=True)
    assert equal(got_g, want_g)
    unit = torch.autograd.grad(want, [p for p in ref if p is not None], torch.eye(5, device=DEV)[0].expand(B, 5))
    assert equal([g for g, p in zip(out[1:], preds) if p is not None], unit)


@pytest.mark.parametrize("rank,per_class_max", [("class", 0), ("score", 0), ("score", 5)])
def test_detection_tail(rank, per_class_max):
    B, R = 2, 300
    rois, cnt = region.rpn_proposals(*rpn_head(B, 50), image_hw=PADDED, mode="test")
    hc, hr = synth.head_outputs(51, B * R, NC)
    hc, hr = torch.from_numpy(hc).to(DEV), torch.from_numpy(hr).to(DEV)
    prob, boxes = frr.decode_classwise(hc, hr, rois.reshape(-1, 4), NC)
    assert equal((prob, boxes), ops.decode_classwise(hc, hr, rois.reshape(-1, 4), NC))
    for cap in (None, 200):
        det = frr.class_nms(prob.view(B, R, NC), boxes.view(B, R, 4 * NC), NC, 0.05, 0.3, cnt, cap)
        assert equal(det, ops.class_nms(prob.view(B, R, NC), boxes.view(B, R, 4 * NC), NC, 0.05, 0.3, roi_count=cnt, cap=cap))
    wh = torch.tensor([[1000.0, 600.0], [480.0, 320.0]], device=DEV)
    for image_wh, xywh in ((None, False), (wh, True)):
        got = frr.pack_detections(*det, 100, image_wh, xywh, rank, per_class_max)
        assert equal(got, ops.pack_detections(*det, 100, image_wh=image_wh, xywh=xywh, rank=rank, per_class_max=per_class_max))


def test_multiscale_roi_align():
    fs, r5 = synth.pyramid_inputs()
    fs = [torch.from_numpy(f).to(DEV) for f in fs]
    r5 = torch.from_numpy(r5).to(DEV)
    scales, k_min, k_max = ops.infer_scales(fs, [(256, 320)])
    x = [f.clone().requires_grad_(True) for f in fs]
    out, levels, per = frr.multiscale_roi_align(x, r5, 7, 7, 2, scales, k_min, k_max, 224.0, 4)
    y = [f.clone().requires_grad_(True) for f in fs]
    want, wlev = ops.multiscale_roi_align(y, r5, [(256, 320)], 7, 2, return_levels=True)
    assert torch.equal(out, want) and torch.equal(levels, wlev)
    go = torch.randn_like(out)
    with deterministic():
        assert equal(torch.autograd.grad(out, x, go), torch.autograd.grad(want, y, go))


# ------------------------------------------------------------------------------------------------
# opcheck
# ------------------------------------------------------------------------------------------------
def _opcheck_cases():
    B = len(SIZES)
    hw = hw_dev(SIZES)
    cls, reg = rpn_head(B, 60)
    rois, cnt = region.rpn_proposals(cls, reg, image_hw=hw, grid_hw=GRID, mode="test")
    r5 = ops.rois5(rois, cnt, GRID, image_hw=hw)
    r5 = r5[live(r5)].contiguous()                       # no masked rois: every output row is written
    f = feats(B, 61)
    gt, gc, gl = gt_batch(B, 5, 62)
    props, pcnt = region.rpn_proposals(cls, reg, image_hw=hw, grid_hw=GRID, mode="train")
    mt = state(63).state
    anchors = ops.anchors_pyramid([(PADDED[0] // s, PADDED[1] // s) for s in (4, 8, 16, 32, 64)], PADDED, DEV)
    g = torch.Generator().manual_seed(64)
    fc = torch.randn((1, anchors.shape[0], 2), generator=g).to(DEV)
    fr = (torch.randn((1, anchors.shape[0], 4), generator=g) * 0.2).to(DEV)
    d = synth.loss_inputs(N=500, S=32, C=5, n_pos=10, n_neg=50, frc_pos=8)
    L = {k: torch.from_numpy(v[None]).to(DEV) for k, v in d.items()}
    hc, hr = (torch.from_numpy(a).to(DEV) for a in synth.head_outputs(65, B * 300, NC))
    prob, boxes = ops.decode_classwise(hc, hr, rois.reshape(-1, 4), NC)
    det = ops.class_nms(prob.view(B, 300, NC), boxes.view(B, 300, 4 * NC), NC, 0.05, 0.3, roi_count=cnt)
    fs, pr5 = synth.pyramid_inputs()
    fs = [torch.from_numpy(a).to(DEV).requires_grad_(True) for a in fs]
    scales, k_min, k_max = ops.infer_scales(fs, [(256, 320)])
    rg = lambda t: t.clone().requires_grad_(True)        # noqa: E731
    return [
        (frr.rpn_proposals_sized, (cls, reg, hw, *GRID, 6000, 300, 0.7, ops._MIN_SIZE)),
        (frr.rpn_proposals_anchored, (fc, fr, anchors, 2000, 500, 0.7, 0.01)),
        (frr.rois5, (rois, cnt, *GRID, hw, 16)),
        (frr.rois5, (rois, None, *GRID, None, 16)),
        (frr.roi_pool_sized, (f.clone().requires_grad_(True), r5, hw, 1.0, 7, 7, 16)),
        (frr.make_targets, (gt, gc, gl, props, pcnt, mt, *PADDED, hw)),
        (frr.make_targets, (gt, None, gl, props, pcnt, mt, *PADDED, None)),
        (frr.rpn_targets, (gt, gc, mt, None, *PADDED, hw, "vgg")),
        (frr.rpn_targets, (gt[:1], gc[:1], mt, anchors, 0, 0, None, "fpn")),
        (frr.frcnn_targets, (props, pcnt, gt, gc, gl, mt, "fpn")),
        (frr.region_loss, (rg(L["rpn_cls"]), rg(L["rpn_reg"]), L["rpn_tcls"], L["rpn_treg"], rg(L["frc_cls"]),
                           rg(L["frc_reg"]), L["frc_tcls"], L["frc_treg"])),
        (frr.region_loss, (None, None, None, None, rg(L["frc_cls"]), rg(L["frc_reg"][:, :, 0]), L["frc_tcls"], L["frc_treg"])),
        (frr.decode_classwise, (hc, hr, rois.reshape(-1, 4), NC)),
        (frr.class_nms, (prob.view(B, 300, NC), boxes.view(B, 300, 4 * NC), NC, 0.05, 0.3, cnt, None)),
        (frr.pack_detections, (*det, 100, None, False, "score", 0)),
        (frr.pack_detections, (*det, 50, torch.full((B, 2), 500.0, device=DEV), True, "class", 0)),
        (frr.multiscale_roi_align, (fs, torch.from_numpy(pr5).to(DEV), 7, 7, 2, scales, k_min, k_max, 224.0, 4)),
    ]


def test_opcheck():
    with deterministic():        # the RoI backward ops then give the same bits on every run
        for op, args in _opcheck_cases():
            torch.library.opcheck(op, args, test_utils=OPCHECK)


# ------------------------------------------------------------------------------------------------
# whole steps under torch.compile
# ------------------------------------------------------------------------------------------------
def predict_inputs(seed, sizes):
    B = len(sizes)
    cls, reg = rpn_head(B, seed)
    return feats(B, seed + 1), cls, reg, hw_dev(sizes)


def predict(*a):
    return region_steps.predict(*a, grid=GRID, NC=NC)


def check_predict(got, want):
    packed, pc, rois, cnt = got
    assert equal((packed, pc, rois, cnt), want)


@pytest.mark.parametrize("backend", ["aot_eager", "inductor"])
def test_compiled_predict_equals_eager_and_launches_the_same_kernels(backend):
    torch._dynamo.reset()
    w = head_weights(70)
    step = torch.compile(predict, backend=backend, fullgraph=True)
    for seed, sizes in ((71, SIZES), (72, SIZES2)):
        x = predict_inputs(seed, sizes)
        check_predict(step(*x, *w), predict(*x, *w))
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    predict(*x, *w)
    n_eager = _lib.launch_count() - n0
    n0 = _lib.launch_count()
    step(*x, *w)
    assert _lib.launch_count() - n0 == n_eager > 0


def train_inputs(seed, sizes, sized):
    B = len(sizes)
    cls, reg = rpn_head(B, seed)
    hw = hw_dev(sizes) if sized else None
    props, pcnt = region.rpn_proposals(cls, reg, image_hw=hw if hw is not None else PADDED, grid_hw=GRID, mode="train")
    gt, gc, gl = gt_batch(B, 6, seed + 1)
    return feats(B, seed + 2), cls, reg, gt, gc, gl, props, pcnt, hw


def run_train(fn, x, w, mt0):
    f, cls, reg, gt, gc, gl, props, pcnt, hw = x
    f, cls, reg = (t.clone().requires_grad_(True) for t in (f, cls, reg))
    mt = mt0.clone()
    loss, t, r5 = fn(f, cls, reg, gt, gc, gl, props, pcnt, mt, hw, *w)
    loss[:, 0].sum().backward()
    return loss, t, r5, mt, f.grad, cls.grad, reg.grad


def train(*a):
    return region_steps.train(*a, padded_hw=PADDED, NC=NC)


@pytest.mark.parametrize("backend", ["aot_eager", "inductor"])
@pytest.mark.parametrize("sized", [False, True])
def test_compiled_train_equals_eager_and_launches_the_same_kernels(backend, sized):
    torch._dynamo.reset()
    w = head_weights(80)
    mt0 = state(81).state
    step = torch.compile(train, backend=backend, fullgraph=True)
    for seed in (82, 83):
        x = train_inputs(seed, SIZES, sized)
        for det in (True, False):
            with deterministic(det):
                got, want = run_train(step, x, w, mt0), run_train(train, x, w, mt0)
            loss, t, r5, mt, g_feat, g_cls, g_reg = got
            assert equal((loss, t, r5, mt), want[:4])
            assert equal((g_cls, g_reg), want[5:])
            if det:
                assert torch.equal(g_feat, want[4])
            else:
                assert float((g_feat - want[4]).abs().max()) <= 1e-5 * float(want[4].abs().max())
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    run_train(train, x, w, mt0)
    n_eager = _lib.launch_count() - n0
    n0 = _lib.launch_count()
    run_train(step, x, w, mt0)
    assert _lib.launch_count() - n0 == n_eager > 0


def test_reduce_overhead_predict_replays_new_inputs_and_sizes():
    """CUDA graph trees: the captured step is replayed on new features, head outputs and per-image sizes written into the
    same tensors; every replay equals the eager step on those inputs."""
    torch._dynamo.reset()
    w = head_weights(90)
    x = predict_inputs(91, SIZES)
    step = torch.compile(predict, mode="reduce-overhead", fullgraph=True)
    for _ in range(3):                                   # warm-up, record
        step(*x, *w)
    runs = [(92, SIZES2), (93, SIZES), (94, [(160, 480), (320, 320), (48, 64)])]
    for seed, sizes in runs:
        new = predict_inputs(seed, sizes)
        for dst, src in zip(x, new):
            dst.copy_(src)
        got = [t.clone() for t in step(*x, *w)]
        check_predict(got, predict(*x, *w))


@pytest.mark.parametrize("backend", ["aot_eager", "inductor"])
def test_compiled_multiscale_roi_align_equals_eager(backend):
    torch._dynamo.reset()
    fs, r5 = synth.pyramid_inputs()
    r5 = torch.from_numpy(r5).to(DEV)
    scales, k_min, k_max = ops.infer_scales([torch.from_numpy(f) for f in fs], [(256, 320)])

    def fwd(r5, *feats):
        return frr.multiscale_roi_align(list(feats), r5, 7, 7, 2, scales, k_min, k_max, 224.0, 4)[0]

    step = torch.compile(fwd, backend=backend, fullgraph=True)
    go = torch.randn((r5.shape[0], fs[0].shape[1], 7, 7), device=DEV)
    with deterministic():
        x = [torch.from_numpy(f).to(DEV).requires_grad_(True) for f in fs]
        y = [torch.from_numpy(f).to(DEV).requires_grad_(True) for f in fs]
        out = step(r5, *x)
        want = ops.multiscale_roi_align(y, r5, [(256, 320)], 7, 2)
        assert torch.equal(out, want)
        assert equal(torch.autograd.grad(out, x, go), torch.autograd.grad(want, y, go))
