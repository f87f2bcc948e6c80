"""Mixed-size batches: images padded to one feature grid, per-image sizes given as an int32 [B,2] device tensor.

Every image of a sized call must get exactly what the uniform path gives for that image alone at its own size, on the
cropped inputs (indices mapped by (y * grid_w + x) * A + a <-> (y * fw + x) * A + a).  The padding cells of the batch
hold NaN, +-inf and huge values, so a kernel that reads or clips against padding shows up as a mismatch.
"""
import numpy as np
import pytest
import torch

from faster_rcnn_pytorch_b200 import ops, region, targets

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
S = 16
A = 9
GRID = (20, 30)                    # padded grid in cells: a 320 x 480 batch
MAX_HW = (GRID[0] * S, GRID[1] * S)
# one image filling the grid, one half as wide as the grid, VOC-like aspect ratios, a 1-cell and a 0-cell image
SIZES = [(320, 480), (320, 240), (240, 320), (300, 470), (16, 16), (8, 480), (200, 100)]
SAME = [(240, 352)] * 4            # every image the same size: the sized path must equal the uniform one bit for bit
BAD = [(99999, 99999), (-16, 64), (320, 480)]   # out of range: clamped to the grid / empty, never a fault


def cells(hw):
    return max(hw[0] // S, 0), max(hw[1] // S, 0)


def dev_hw(sizes):
    return torch.tensor(sizes, dtype=torch.int32, device=DEV)


def fill_padding(x, sizes, grid, seed):
    """x [B, grid_h * grid_w * A, k]: padding cells of each image <- NaN, +-inf and 1e30 (in place)."""
    B, k = x.shape[0], x.shape[-1]
    v = x.view(B, grid[0], grid[1], A, k)
    g = torch.Generator().manual_seed(seed)
    junk = torch.tensor([float("nan"), float("inf"), -float("inf"), 1e30, -1e30], device=x.device)
    for b, hw in enumerate(sizes):
        fh, fw = min(cells(hw)[0], grid[0]), min(cells(hw)[1], grid[1])
        mask = torch.ones(grid, dtype=torch.bool, device=x.device)
        mask[:fh, :fw] = False
        n = int(mask.sum()) * A * k
        pick = torch.randint(0, 5, (n,), generator=g).to(x.device)
        v[b][mask] = junk[pick].view(-1, A, k)
    return x


def head(B, grid, seed, sizes):
    g = torch.Generator().manual_seed(seed)
    N = grid[0] * grid[1] * A
    cls = torch.randn((B, N, 2), generator=g).to(DEV)
    reg = (torch.randn((B, N, 4), generator=g) * 0.2).to(DEV)
    return fill_padding(cls, sizes, grid, seed + 1), fill_padding(reg, sizes, grid, seed + 2)


def crop(x, b, hw, grid):
    """image b's own [1, fh * fw * A, k] inputs out of the padded [B, N, k] tensor"""
    fh, fw = cells(hw)
    k = x.shape[-1]
    return x[b].view(grid[0], grid[1], A, k)[:fh, :fw].reshape(1, fh * fw * A, k).contiguous()


def crop_n(x, b, hw, grid):
    """the same for a [B, N] tensor"""
    return crop(x.unsqueeze(-1), b, hw, grid)[..., 0]


def to_own(idx, hw, grid):
    """padded anchor indices -> the image's own indices"""
    cell, a = idx // A, idx % A
    y, x = cell // grid[1], cell % grid[1]
    return (y * cells(hw)[1] + x) * A + a


def gt_batch(B, G, seed):
    rs = np.random.RandomState(seed)
    xy1 = rs.uniform(0.0, 0.7, (B, G, 2))
    wh = rs.uniform(0.05, 0.3, (B, G, 2))
    gt = torch.from_numpy(np.concatenate([xy1, xy1 + wh], axis=2).astype(np.float32)).to(DEV)
    count = torch.from_numpy(rs.randint(1, G + 1, B).astype(np.int32)).to(DEV)
    labels = torch.from_numpy(rs.randint(0, 20, (B, G)).astype(np.int64)).to(DEV)
    return gt, count, labels


def live(rois5):
    """rows of rois with a batch index: the RoI kernels leave the output rows of masked rois (index -1) unwritten"""
    return rois5[:, 0] >= 0


def real(sizes):
    return [b for b, hw in enumerate(sizes) if cells(hw)[0] > 0 and cells(hw)[1] > 0]


# ------------------------------------------------------------------------------------------------
# decode, top-k, NMS
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("logits", [True, False])
def test_decode_per_image(logits):
    B = len(SIZES)
    cls, reg = head(B, GRID, 11, SIZES)
    if not logits:
        cls = fill_padding(torch.rand((B, cls.shape[1], 1), device=DEV), SIZES, GRID, 5)[..., 0].contiguous()
    boxes, scores, valid = ops.rpn_decode(reg, cls, image_hw=dev_hw(SIZES), grid_hw=GRID)
    for b, hw in enumerate(SIZES):
        fh, fw = cells(hw)
        pad = torch.ones(GRID, dtype=torch.bool, device=DEV)
        pad[:fh, :fw] = False
        assert int(valid[b].view(*GRID, A)[pad].sum()) == 0
        if fh * fw == 0:
            continue
        c = crop(cls, b, hw, GRID) if logits else crop_n(cls, b, hw, GRID)
        rb, rs_, rv = ops.rpn_decode(crop(reg, b, hw, GRID), c, image_hw=hw)
        torch.testing.assert_close(crop(boxes, b, hw, GRID), rb, rtol=1e-5, atol=0)
        torch.testing.assert_close(crop_n(scores, b, hw, GRID), rs_, rtol=1e-5, atol=0)
        assert torch.equal(crop_n(valid, b, hw, GRID), rv)


@pytest.mark.parametrize("mode", ["train", "test"])
def test_proposals_per_image(mode):
    B = len(SIZES)
    cls, reg = head(B, GRID, 21, SIZES)
    out = region.rpn_proposals(cls, reg, image_hw=dev_hw(SIZES), grid_hw=GRID, mode=mode, return_all=True)
    for b, hw in enumerate(SIZES):
        if b not in real(SIZES):
            assert int(out["count"][b]) == 0 and int(out["topk"]["count"][b]) == 0
            assert not out["rois"][b].any()
            continue
        ref = region.rpn_proposals(crop(cls, b, hw, GRID), crop(reg, b, hw, GRID), image_hw=hw, mode=mode, return_all=True)
        n = int(ref["topk"]["count"][0])
        assert int(out["topk"]["count"][b]) == n
        assert torch.equal(to_own(out["topk"]["idx"][b, :n].long(), hw, GRID), ref["topk"]["idx"][0, :n].long())
        assert torch.equal(out["topk"]["cidx"][b, :n], ref["topk"]["cidx"][0, :n])
        assert torch.equal(out["count"][b], ref["count"][0])
        assert torch.equal(out["keep"][b], ref["keep"][0])
        assert torch.equal(out["rois"][b], ref["rois"][0])


def test_same_sizes_equal_uniform_path():
    B, hw = len(SAME), SAME[0]
    grid = cells(hw)
    g = torch.Generator().manual_seed(3)
    N = grid[0] * grid[1] * A
    cls = torch.randn((B, N, 2), generator=g).to(DEV)
    reg = (torch.randn((B, N, 4), generator=g) * 0.2).to(DEV)
    sized = region.rpn_proposals(cls, reg, image_hw=dev_hw(SAME), grid_hw=grid, return_all=True)
    uni = region.rpn_proposals(cls, reg, image_hw=hw, return_all=True)
    for key in ("rois", "count", "keep", "boxes", "scores", "valid"):
        assert torch.equal(sized[key], uni[key]), key
    gt, gtc, _ = gt_batch(B, 6, 4)
    torch.manual_seed(5)
    a = targets.rpn_targets(gt, gtc, image_hw=dev_hw(SAME), grid_hw=grid)
    torch.manual_seed(5)
    u = targets.rpn_targets(gt, gtc, image_hw=hw)
    assert torch.equal(a[0], u[0]) and torch.equal(a[1], u[1])
    feat = torch.randn((B, 16, *grid), device=DEV)
    r5s = ops.rois5(sized["rois"], sized["count"], grid, image_hw=dev_hw(SAME))
    r5u = ops.rois5(uni["rois"], uni["count"], grid)
    assert torch.equal(r5s, r5u)
    os_, as_ = ops.roi_pool_forward(feat, r5s, image_hw=dev_hw(SAME))
    ou, au = ops.roi_pool_forward(feat, r5u)
    m = live(r5u)
    assert torch.equal(os_[m], ou[m]) and torch.equal(as_[m], au[m])


def test_out_of_range_sizes_are_clamped():
    B = len(BAD)
    cls, reg = head(B, GRID, 31, [(320, 480)] * B)
    hw = dev_hw(BAD)
    boxes, scores, valid = ops.rpn_decode(reg, cls, image_hw=hw, grid_hw=GRID)
    rois, count = region.rpn_proposals(cls, reg, image_hw=hw, grid_hw=GRID)
    torch.cuda.synchronize()
    assert int(valid[1].sum()) == 0 and int(count[1]) == 0 and not rois[1].any()
    assert int(count[0]) > 0 and torch.isfinite(rois).all()
    gt, gtc, _ = gt_batch(B, 4, 6)
    labels, _ = targets.rpn_targets(gt, gtc, image_hw=hw, grid_hw=GRID)
    assert (labels[1] == -1).all()
    r5 = ops.rois5(rois, count, GRID, image_hw=hw)
    assert (r5.view(B, -1, 5)[1, :, 0] == -1).all()
    feat = torch.randn((B, 8, *GRID), device=DEV)
    out, arg = ops.roi_pool_forward(feat, r5, image_hw=hw)
    torch.cuda.synchronize()
    assert int(arg[live(r5)].max()) < GRID[0] * GRID[1]
    with pytest.raises(ValueError):
        ops.rpn_decode(reg, cls, image_hw=BAD, grid_hw=GRID)       # host sizes are checked against the grid


# ------------------------------------------------------------------------------------------------
# RPN targets and sampling
# ------------------------------------------------------------------------------------------------
def _per_image_targets(gt, gtc, sizes, generator_seed=None, seed=0):
    """the reference stream: one image at a time, at its own size"""
    torch.manual_seed(seed)
    gen = targets.DeviceGenerator(DEV) if generator_seed else None
    res = {}
    for b, hw in enumerate(sizes):
        if b not in real(sizes):
            continue
        res[b] = targets.rpn_targets(gt[b:b + 1], gtc[b:b + 1], image_hw=hw, generator=gen)
    return res, gen


@pytest.mark.parametrize("device_sampling", [False, True])
def test_rpn_targets_per_image(device_sampling):
    B = len(SIZES)
    gt, gtc, _ = gt_batch(B, 8, 41)
    ref, rgen = _per_image_targets(gt, gtc, SIZES, device_sampling, seed=123)
    ref_state = torch.get_rng_state()
    torch.manual_seed(123)
    gen = targets.DeviceGenerator(DEV) if device_sampling else None
    labels, reg = targets.rpn_targets(gt, gtc, image_hw=SIZES, grid_hw=GRID, generator=gen)
    if device_sampling:
        assert torch.equal(gen.state, rgen.state)
    else:
        assert torch.equal(torch.get_rng_state(), ref_state)
    for b, hw in enumerate(SIZES):
        fh, fw = cells(hw)
        pad = torch.ones(GRID, dtype=torch.bool, device=DEV)
        pad[:fh, :fw] = False
        assert (labels[b].view(*GRID, A)[pad] == -1).all()
        assert not reg[b].view(*GRID, A, 4)[pad].any()
        if b in ref:
            assert torch.equal(crop_n(labels, b, hw, GRID), ref[b][0])
            assert torch.equal(crop(reg, b, hw, GRID), ref[b][1])


# ------------------------------------------------------------------------------------------------
# RoIPool forward / backward
# ------------------------------------------------------------------------------------------------
# (name, grid in cells, stride, sizes, C, output size, expected forward kernel, channels_last)
ROI_CASES = [
    ("flat", GRID, 16, SIZES, 64, (7, 7), "pool_fwd_flat", False),
    ("flat_nhwc", GRID, 16, SIZES, 64, (7, 7), "pool_fwd_flat", True),
    ("planes", GRID, 16, SIZES, 16, (14, 14), "fwd_planes", False),
    ("direct", (200, 336), 1, [(200, 336), (200, 168), (120, 300), (1, 1), (0, 50)], 4, (3, 5), "fwd_direct", False),
]


def _rois(sizes, per_image, seed):
    """normalised rois per image, a third of them clamped to the right / bottom edge (x2 = 1 or y2 = 1)"""
    rs = np.random.RandomState(seed)
    B = len(sizes)
    x1 = rs.uniform(0.0, 0.9, (B, per_image))
    y1 = rs.uniform(0.0, 0.9, (B, per_image))
    x2 = np.minimum(x1 + rs.uniform(0.02, 0.8, (B, per_image)), 1.0)
    y2 = np.minimum(y1 + rs.uniform(0.02, 0.8, (B, per_image)), 1.0)
    x2[:, ::3] = 1.0
    y2[:, 1::3] = 1.0
    return torch.from_numpy(np.stack([x1, y1, x2, y2], axis=2).astype(np.float32)).to(DEV)


@pytest.mark.parametrize("case", ROI_CASES, ids=[c[0] for c in ROI_CASES])
def test_roi_pool_per_image(case):
    _, grid, stride, sizes, C, out_size, kernel, nhwc = case
    B, R = len(sizes), 24
    rois = _rois(sizes, R, 51)
    count = torch.full((B,), R, dtype=torch.int32, device=DEV)
    hw = dev_hw(sizes)
    assert ops.roi_variant("roi_pool_fwd", B * R, B, C, *grid, output_size=out_size)["kernel"] == kernel
    g = torch.Generator().manual_seed(52)
    feat = torch.randn((B, C, *grid), generator=g).to(DEV)
    for b, s in enumerate(sizes):                                    # padding: huge values, +inf
        fh, fw = (max(s[0] // stride, 0), max(s[1] // stride, 0))
        feat[b, :, fh:, :] = 1e30
        feat[b, :, :, fw:] = float("inf")
    if nhwc:
        feat = feat.to(memory_format=torch.channels_last)
    r5 = ops.rois5(rois, count, grid, image_hw=hw, stride=stride)
    out, arg = ops.roi_pool_forward(feat, r5, out_size, image_hw=hw, stride=stride)
    go = torch.randn(out.shape, generator=g).to(DEV)
    gin = ops.roi_pool_backward(go, arg, r5, tuple(feat.shape), channels_last=nhwc, deterministic=False)
    gdet = ops.roi_pool_backward(go, arg, r5, tuple(feat.shape), channels_last=nhwc, deterministic=True, image_hw=hw,
                                 stride=stride)
    K = B * R
    out, arg, go = out.view(B, R, -1), arg.view(B, R, -1), go.view(B, R, -1)
    for b, s in enumerate(sizes):
        fh, fw = (max(s[0] // stride, 0), max(s[1] // stride, 0))
        pad = torch.ones(grid, dtype=torch.bool, device=DEV)
        pad[:fh, :fw] = False
        assert not gin[b][:, pad].any() and not gdet[b][:, pad].any()
        if fh * fw == 0:
            assert (r5.view(B, R, 5)[b, :, 0] == -1).all()
            continue
        fb = feat[b:b + 1, :, :fh, :fw]
        fb = fb.contiguous(memory_format=torch.channels_last) if nhwc else fb.contiguous()
        rb = ops.rois5(rois[b:b + 1].contiguous(), count[b:b + 1], (fh, fw))
        ro, ra = ops.roi_pool_forward(fb, rb, out_size)
        assert torch.equal(out[b], ro.view(R, -1))
        own = torch.where(arg[b] >= 0, (arg[b] // grid[1]) * fw + arg[b] % grid[1], arg[b])
        assert torch.equal(own, ra.view(R, -1))
        gob = go[b].reshape(ro.shape).contiguous()
        rg = ops.roi_pool_backward(gob, ra, rb, tuple(fb.shape), channels_last=nhwc, deterministic=False)
        tol = 1e-5 * float(rg.abs().max())
        torch.testing.assert_close(gin[b, :, :fh, :fw], rg[0], rtol=0, atol=tol)
        rd = ops.roi_pool_backward(gob, ra, rb, tuple(fb.shape), channels_last=nhwc, deterministic=True)
        assert torch.equal(gdet[b, :, :fh, :fw], rd[0])
    assert K == r5.shape[0]


def test_roi_pool_autograd_carries_the_extent():
    B, C = len(SIZES), 16
    rois = _rois(SIZES, 10, 61)
    hw = dev_hw(SIZES)
    r5 = ops.rois5(rois, None, GRID, image_hw=hw)
    feat = torch.randn((B, C, *GRID), device=DEV)
    feat[:, :, 15:, :] = 1e30
    feat.requires_grad_(True)
    boxes = r5[r5[:, 0] >= 0]
    out = ops.roi_pool(feat, boxes, 7, image_hw=hw)
    ref, arg = ops.roi_pool_forward(feat.detach(), boxes, image_hw=hw)
    assert torch.equal(out.detach(), ref)
    assert torch.equal(out.grad_fn.saved_tensors[2], hw)      # the backward gets the forward's sizes
    go = torch.randn_like(out)
    torch.use_deterministic_algorithms(True)
    try:
        (g,) = torch.autograd.grad(out, feat, go)
    finally:
        torch.use_deterministic_algorithms(False)
    assert torch.equal(g, ops.roi_pool_backward(go, arg, boxes, tuple(feat.shape), deterministic=True, image_hw=hw))


def test_deterministic_backward_clips_to_the_image():
    """an argmax inside a bin's unclipped window but in the padding adds nothing once the window is clipped to the image"""
    B, C = 2, 4
    hw = dev_hw([(320, 480), (320, 240)])                       # image 1: 20 x 15 cells of the 20 x 30 grid
    r5 = torch.tensor([[1.0, 0.0, 0.0, GRID[1] - 1.0, GRID[0] - 1.0]], device=DEV)   # spans the padded map
    go = torch.ones((1, C, 7, 7), device=DEV)
    arg = torch.full((1, C, 7, 7), 25, dtype=torch.int32, device=DEV)   # pixel (0, 25): padding of image 1
    shape = (B, C, *GRID)
    clipped = ops.roi_pool_backward(go, arg, r5, shape, deterministic=True, image_hw=hw)
    unclipped = ops.roi_pool_backward(go, arg, r5, shape, deterministic=True)
    assert (unclipped[1, :, 0, 25] > 0).all()
    assert not clipped.any()


# ------------------------------------------------------------------------------------------------
# loss on a padded batch
# ------------------------------------------------------------------------------------------------
def test_region_loss_with_padding():
    sizes = [s for s in SIZES if cells(s)[0] * cells(s)[1] > 0]
    B = len(sizes)
    cls, reg = head(B, GRID, 71, sizes)
    gt, gtc, _ = gt_batch(B, 8, 72)
    torch.manual_seed(9)
    tc, tr = targets.rpn_targets(gt, gtc, image_hw=sizes, grid_hw=GRID)
    cls.requires_grad_(True)
    reg.requires_grad_(True)
    loss = ops.region_loss(cls, reg, tc, tr)
    gc, gr = torch.autograd.grad(loss[:, 0].sum(), (cls, reg))
    for b, hw in enumerate(sizes):
        fh, fw = cells(hw)
        pad = torch.ones(GRID, dtype=torch.bool, device=DEV)
        pad[:fh, :fw] = False
        assert not gc[b].view(*GRID, A, 2)[pad].any() and not gr[b].view(*GRID, A, 4)[pad].any()
        c, r = crop(cls.detach(), b, hw, GRID).requires_grad_(True), crop(reg.detach(), b, hw, GRID).requires_grad_(True)
        lb = ops.region_loss(c, r, crop_n(tc, b, hw, GRID), crop(tr, b, hw, GRID))
        rc, rr = torch.autograd.grad(lb[:, 0].sum(), (c, r))
        # an image with nothing sampled has the reference's 0 / 0 (NaN) RPN losses, alone and in the batch alike
        nan = torch.isnan(lb[0])
        assert torch.equal(torch.isnan(loss[b]), nan)
        # per-thread sums differ in order between the padded and the cropped layout
        torch.testing.assert_close(loss[b].detach()[~nan], lb[0].detach()[~nan], rtol=1e-5, atol=0)
        assert torch.equal(crop(gc, b, hw, GRID), rc) and torch.equal(crop(gr, b, hw, GRID), rr)


# ------------------------------------------------------------------------------------------------
# plans, graphs, pipeline
# ------------------------------------------------------------------------------------------------
MIX1 = [(320, 480), (320, 240), (240, 320), (16, 16)]
MIX2 = [(300, 400), (8, 480), (320, 480), (192, 288)]


def test_infer_plan_graph_replays_two_size_mixes():
    B, C = 4, 32
    plan = region.InferPlan(B, MAX_HW, 21, DEV)
    hw = dev_hw(MIX1)
    cls, reg = head(B, GRID, 81, [MAX_HW] * B)
    feat = torch.randn((B, C, *GRID), device=DEV)
    graph, (pooled, rois, cnt) = plan.capture_pool(feat, cls, reg, image_hw=hw)
    eager = region.InferPlan(B, MAX_HW, 21, DEV)
    for mix, seed in ((MIX1, 82), (MIX2, 83)):
        hw.copy_(dev_hw(mix))
        c2, r2 = head(B, GRID, seed, mix)
        cls.copy_(c2)
        reg.copy_(r2)
        graph.replay()
        ep, er, ec = eager.pool(feat, cls, reg, image_hw=dev_hw(mix))
        m = live(eager.rois5)
        assert torch.equal(cnt, ec) and torch.equal(rois, er) and torch.equal(plan.rois5, eager.rois5)
        assert torch.equal(pooled[m], ep[m])
        for b, s in enumerate(mix):           # and each image as alone
            if b not in real(mix):
                assert int(cnt[b]) == 0
                continue
            ref, rc = region.rpn_proposals(crop(cls, b, s, GRID), crop(reg, b, s, GRID), image_hw=s, mode="test")
            assert torch.equal(rois[b], ref[0]) and torch.equal(cnt[b], rc[0])


def test_train_plan_graph_replays_two_size_mixes():
    B, C = 4, 32
    gt, gtc, glab = gt_batch(B, 6, 91)
    feat = torch.randn((B, C, *GRID), device=DEV)
    cls, reg = head(B, GRID, 92, MIX1)
    props, pcount = region.rpn_proposals(cls, reg, image_hw=dev_hw(MIX1), grid_hw=GRID)
    torch.manual_seed(93)
    plan = region.TrainPlan(B, MAX_HW, DEV)
    eager = region.TrainPlan(B, MAX_HW, DEV)
    hw = dev_hw(MIX1)
    graph, (t, pooled) = plan.capture_targets_and_pool(feat, gt, glab, props, pcount, image_hw=hw)
    go = torch.randn(pooled.shape, device=DEV)
    bgraph, grad = plan.capture_pool_backward(go)
    for mix in (MIX1, MIX2):
        hw.copy_(dev_hw(mix))
        eager.generator.state.copy_(plan.generator.state)
        graph.replay()
        bgraph.replay()
        et, ep = eager.targets_and_pool(feat, gt, glab, props, pcount, image_hw=dev_hw(mix))
        eg = eager.pool_backward(go)
        assert torch.equal(plan.generator.state, eager.generator.state)
        for key in ("rpn_cls", "rpn_reg", "frcnn_cls", "frcnn_reg", "sample_rois", "n_samples"):
            assert torch.equal(t[key], et[key]), key
        m = live(eager.rois5)
        assert torch.equal(plan.rois5, eager.rois5) and torch.equal(pooled[m], ep[m])
        torch.testing.assert_close(grad, eg, rtol=0, atol=1e-5 * float(eg.abs().max()))
        for b, s in enumerate(mix):
            fh, fw = cells(s)
            assert (t["rpn_cls"][b].view(*GRID, A)[fh:] == -1).all() and (t["rpn_cls"][b].view(*GRID, A)[:, fw:] == -1).all()
            assert not grad[b][:, fh:].any() and not grad[b][:, :, fw:].any()


def test_proposal_pipeline_four_in_flight():
    B, depth = 4, 4
    N = GRID[0] * GRID[1] * A
    pipe = region.ProposalPipeline(B, N, DEV, depth=depth, image_hw=MAX_HW)
    mixes = [MIX1, MIX2, MIX2[::-1], MIX1[::-1]]
    batches = [(head(B, GRID, 100 + i, m), dev_hw(m)) for i, m in enumerate(mixes)]
    tickets = [pipe.submit(c, r, image_hw=h) for (c, r), h in batches]
    for t, ((c, r), h) in zip(tickets, batches):
        rois, count = pipe.result(t)
        ref, rc = region.rpn_proposals(c, r, image_hw=h, grid_hw=GRID)
        assert torch.equal(rois, ref) and torch.equal(count, rc)
    (c, r), _ = batches[1]
    t = pipe.submit(c, r, image_hw=MIX2)                          # host sizes are checked and copied
    rois, count = pipe.result(t)
    ref, rc = region.rpn_proposals(c, r, image_hw=MIX2, grid_hw=GRID)
    assert torch.equal(rois, ref) and torch.equal(count, rc)
