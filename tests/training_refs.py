"""Plain high-precision references for the training half of the region stage: the fused region loss in float64 (with
per-element error bounds for the fp32 kernel), the target encoding in float64, and the host searches that build
threshold-exact IoU pairs and cross-slab IoU ties.  Shared by the GPU tests and their CPU self-checks."""
import functools
import math

import numpy as np
import torch

f32 = np.float32
U = 2.0 ** -24                       # unit roundoff of fp32
TINY = 1e-30                         # below the scale of any nonzero term here
LOSS_THREADS = 1024                  # loss.cu: one CTA of 1024 threads per image
WARPS = LOSS_THREADS // 32
RPN_BETA, FRCNN_BETA = f32(1 / 9), f32(1.0)
WORST = {}                           # largest error / bound ratio seen per quantity (printed by the GPU tests)


# ------------------------------------------------------------------------------------------------
# region loss
# ------------------------------------------------------------------------------------------------
def _sl1(p32, q32, beta):
    """SmoothL1 of float64 leaves made from the fp32 predictions: the branch is taken on the fp32 difference against
    fp32(beta), as the reference's fp32 torch expression does; the value is evaluated in float64."""
    mask = torch.from_numpy(np.abs(p32 - q32) >= f32(beta))
    p = torch.from_numpy(p32.astype(np.float64)).requires_grad_(True)
    d = p - torch.from_numpy(q32.astype(np.float64))
    b = float(f32(beta))
    return p, torch.where(mask, d.abs() - 0.5 * b, 0.5 * d * d / b)


def _ce(l32, t):
    """Cross entropy rows in float64 (with their float64 leaf), the fp32 torch value of each row, and per-row
    magnitudes for the bound: |max logit|, |lse - max|, |target logit|."""
    l = torch.from_numpy(l32.astype(np.float64)).requires_grad_(True)
    tt = torch.from_numpy(np.asarray(t, np.int64))
    r = torch.arange(len(t))
    terms = torch.logsumexp(l, 1) - l[r, tt]
    with np.errstate(all="ignore"):
        fp32 = torch.nn.functional.cross_entropy(torch.from_numpy(l32), tt, reduction="none").numpy()
        ld = l.detach().numpy()
        m = ld.max(1) if ld.size else np.zeros(0)
        mag = np.abs(m) + np.abs(terms.detach().numpy() + ld[r, tt] - m) + np.abs(ld[r, tt])
    return l, terms, fp32, mag


def _grad_scale(k, ld, weight):
    """2u (k + |l_c - max|) (p_c + onehot_c): the exp argument's rounding, expf, the exp sum, the reciprocal and the
    products, relative to the softmax value and the one-hot term (0 where both are 0, also at l_c = -inf)."""
    if not ld.size:
        return np.zeros_like(ld)
    with np.errstate(all="ignore"):
        r = 2 * U * (k + np.abs(ld - ld.max(1, keepdims=True))) * weight
    return np.where(weight > 0, r, 0.0)


def loss_reference(x, upstream=None, rpn_beta=RPN_BETA, frcnn_beta=FRCNN_BETA):
    """One image of ``ops.region_loss`` in float64.  ``x``: rpn_cls [N,2], rpn_reg [N,4], rpn_tcls [N], rpn_treg [N,4],
    frc_cls [S,C], frc_reg [S,CR,4], frc_tcls [S], frc_treg [S,4] (fp32 / int64 numpy; a half may be None).
    A Fast R-CNN class >= C counts in the normaliser and adds no term (see frr_region_loss in include/frr.h).

    Returns dict(loss float64 [5], bound [5], fp32 [5] (the fp32 torch value where it is not finite, else NaN-free
    placeholder), finite [5] bool, grads (four float64 arrays or None), gbound (four arrays or None)) for the upstream
    gradient ``upstream`` [5] (default: the total only)."""
    g = np.asarray([1, 0, 0, 0, 0], np.float64) if upstream is None else np.asarray(upstream, np.float64)
    g32 = np.asarray(g, f32)
    loss = np.zeros(5)
    bound = np.zeros(5)
    fp32 = np.zeros(5)                       # fp32 torch expression of each component (inf / NaN propagate)
    grads, gbound = [None] * 4, [None] * 4
    objective = torch.zeros((), dtype=torch.float64)
    unit = [None] * 4                        # per-element bound on the unit-upstream gradient

    if x.get("rpn_cls") is not None:
        t = np.asarray(x["rpn_tcls"])
        N = len(t)
        valid, pos = np.nonzero(t >= 0)[0], np.nonzero(t > 0)[0]
        nv = float(len(valid))
        l, ce, ce32, mag = _ce(x["rpn_cls"][valid], t[valid])
        p, sl = _sl1(x["rpn_reg"][pos], x["rpn_treg"][pos], rpn_beta)
        with np.errstate(all="ignore"):
            lc = ce.sum() / nv if nv else torch.tensor(float("nan"), dtype=torch.float64)
            lr = sl.sum() / nv if nv else torch.tensor(float("nan"), dtype=torch.float64)
            fp32[1] = np.float32(ce32.sum(dtype=f32)) / f32(nv) if nv else np.nan
            fp32[2] = np.nan if not nv else 0.0
        chain = math.ceil(N / LOSS_THREADS)
        # bound: the terms go through a per-thread chain of ceil(N/1024) (x4 for the four box components), a 5-level
        # warp tree and a 32-warp sequential sum, then one division by the exact count
        d_cls, d_reg = chain + 5 + WARPS, 4 * chain + 5 + WARPS
        cet, slt = ce.detach().numpy(), sl.detach().numpy()
        dd = np.abs(x["rpn_reg"][pos].astype(np.float64) - x["rpn_treg"][pos])
        e_ce = 4 * U * (mag + 9.0)                           # a few ulp per CE term vs |max| + |lse - max| + |target|
        e_sl = 4 * U * (slt + dd + float(rpn_beta))          # a few ulp per SmoothL1 term
        if nv:
            bound[1] = ((d_cls + 2) * U * np.abs(cet).sum() + e_ce.sum()) / nv + 2 * U * abs(float(lc.detach()))
            bound[2] = ((d_reg + 2) * U * np.abs(slt).sum() + e_sl.sum()) / nv + 2 * U * abs(float(lr.detach()))
        loss[1], loss[2] = float(lc.detach()), float(lr.detach())
        if nv:
            objective = objective + (g[0] + g[1]) * lc + (g[0] + g[2]) * lr
        # unit-gradient bounds: CE (e_c / se - onehot) / nv relative to (p_c + onehot); SmoothL1 sign / nv or d / beta / nv
        ld = l.detach().numpy()
        with np.errstate(all="ignore"):
            pr = np.exp(ld - ld.max(1, keepdims=True)) if ld.size else ld
            pr = pr / pr.sum(1, keepdims=True) if ld.size else pr
            oh = np.zeros_like(ld)
            oh[np.arange(len(valid)), t[valid]] = 1
            ub_c = _grad_scale(16, ld, pr + oh) / nv if nv else np.zeros_like(ld)
            ub_r = 4 * U * (1 + np.abs(x["rpn_reg"][pos] - x["rpn_treg"][pos]).astype(np.float64) / float(rpn_beta)) / nv \
                if nv else np.zeros((len(pos), 4))
        unit[0] = (valid, ub_c, l)
        unit[1] = (pos, ub_r, p)

    if x.get("frc_cls") is not None:
        c = np.asarray(x["frc_tcls"])
        S, C = x["frc_cls"].shape
        CR = x["frc_reg"].shape[1]
        use = np.nonzero((c >= 0) & (c < C))[0]
        fpos = np.nonzero((c > 0) & (c < C))[0]
        nf = float((c >= 0).sum())
        l, ce, ce32, mag = _ce(x["frc_cls"][use], c[use])
        rows = x["frc_reg"][fpos, 0 if CR == 1 else c[fpos]]
        p, sl = _sl1(rows, x["frc_treg"][fpos], frcnn_beta)
        with np.errstate(all="ignore"):
            lc = ce.sum() / nf if nf else torch.tensor(float("nan"), dtype=torch.float64)
            lr = sl.sum() / nf if nf else torch.tensor(float("nan"), dtype=torch.float64)
            fp32[3] = np.float32(ce32.sum(dtype=f32)) / f32(nf) if nf else np.nan
            fp32[4] = np.nan if not nf else 0.0
        chain = math.ceil(S / WARPS)                         # lane 0 of warp w sums rows w, w + 32, ...
        d_cls, d_reg = chain + 5 + WARPS, 4 * chain + 5 + WARPS
        cet, slt = ce.detach().numpy(), sl.detach().numpy()
        dd = np.abs(rows.astype(np.float64) - x["frc_treg"][fpos])
        e_ce = 4 * U * (mag + math.ceil(C / 32) + 9.0)       # the C-term exp sum: a lane chain of ceil(C/32) + 5 levels
        e_sl = 4 * U * (slt + dd + float(frcnn_beta))
        if nf:
            bound[3] = ((d_cls + 2) * U * np.abs(cet).sum() + e_ce.sum()) / nf + 2 * U * abs(float(lc.detach()))
            bound[4] = ((d_reg + 2) * U * np.abs(slt).sum() + e_sl.sum()) / nf + 2 * U * abs(float(lr.detach()))
        loss[3], loss[4] = float(lc.detach()), float(lr.detach())
        if nf:
            objective = objective + (g[0] + g[3]) * lc + (g[0] + g[4]) * lr
        ld = l.detach().numpy()
        with np.errstate(all="ignore"):
            mx = ld.max(1, keepdims=True) if ld.size else ld
            pr = np.exp(ld - mx) if ld.size else ld
            pr = pr / pr.sum(1, keepdims=True) if ld.size else pr
            oh = np.zeros_like(ld)
            oh[np.arange(len(use)), c[use]] = 1
            ub_c = _grad_scale(math.ceil(C / 32) + 16, ld, pr + oh) / nf if nf else np.zeros_like(ld)
            ub_r = 4 * U * (1 + np.abs(rows - x["frc_treg"][fpos]).astype(np.float64) / float(frcnn_beta)) / nf \
                if nf else np.zeros((len(fpos), 4))
        unit[2] = (use, ub_c, l)
        unit[3] = (fpos, ub_r, p)

    loss[0] = ((loss[1] + loss[2]) + loss[3]) + loss[4]
    bound[0] = bound[1:].sum() + 3 * U * np.abs(loss[1:]).sum()
    fp32[0] = fp32[1:].sum()
    finite = np.isfinite(fp32)

    if objective.requires_grad:
        objective.backward()
    comp = {0: 1, 1: 2, 2: 3, 3: 4}
    shapes = {0: ("rpn_cls", None), 1: ("rpn_reg", None), 2: ("frc_cls", None), 3: ("frc_reg", None)}
    for j in range(4):
        if unit[j] is None:
            continue
        idx, ub, leaf = unit[j]
        key = shapes[j][0]
        full = np.zeros(x[key].shape, np.float64)
        fb = np.zeros(x[key].shape, np.float64)
        up = float(g32[0] + g32[comp[j]])            # the autograd wrapper adds the two fp32 upstream values
        gr = leaf.grad.numpy() if leaf.grad is not None else np.zeros(leaf.shape)
        # scaling by the upstream: one rounding of (g_total + g_j) and one of the product
        b = abs(up) * ub + 3 * U * np.abs(gr) + TINY
        if j == 3:
            cls = np.asarray(x["frc_tcls"])[idx]
            col = 0 if x["frc_reg"].shape[1] == 1 else cls
            full[idx, col] = gr
            fb[idx, col] = b
        else:
            full[idx] = gr
            fb[idx] = b
        grads[j], gbound[j] = full, fb
    return dict(loss=loss, bound=bound, fp32=fp32, finite=finite, grads=grads, gbound=gbound)


def within(got, ref, bound, what):
    """|got - ref| <= bound per element (float64 reference, bound from the written error model)."""
    got = np.asarray(got)
    err = np.abs(got.astype(np.float64) - ref)
    bad = ~(err <= bound)
    assert not bad.any(), (f"{what}: {int(bad.sum())} elements outside the bound, first at {np.argwhere(bad)[0]}: "
                           f"got {got[bad][0]!r} ref {np.asarray(ref)[bad][0]!r} bound {np.asarray(bound)[bad][0]!r}")
    ratio = float(np.max(err / np.maximum(bound, TINY), initial=0.0))
    key = what.split(" ")[-1]
    WORST[key] = max(WORST.get(key, 0.0), ratio)
    return ratio


def check_loss(got, ref, what="loss"):
    """Components where the reference's fp32 torch expression is NaN / inf must be that value; the rest within the
    float64 bound.  Returns the largest error / bound ratio."""
    got = np.asarray(got, np.float64)
    fin = ref["finite"] & np.isfinite(ref["loss"])
    for q in np.nonzero(~fin)[0]:
        want = ref["fp32"][q] if not ref["finite"][q] else ref["loss"][q]
        assert (np.isnan(want) and np.isnan(got[q])) or got[q] == want, f"{what}[{q}]: got {got[q]!r} want {want!r}"
    return within(got[fin], ref["loss"][fin], ref["bound"][fin], what)


# ------------------------------------------------------------------------------------------------
# target encoding (utils/util.py:22-26,39-43) in float64
# ------------------------------------------------------------------------------------------------
def encode64(gt, box, std=(1.0, 1.0, 1.0, 1.0)):
    """encode(xy_to_cxcy(gt), xy_to_cxcy(box)) / std in float64 from the fp32 corners."""
    g, a = np.asarray(gt, np.float64), np.asarray(box, np.float64)
    gw, gh = g[:, 2] - g[:, 0], g[:, 3] - g[:, 1]
    aw, ah = a[:, 2] - a[:, 0], a[:, 3] - a[:, 1]
    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.stack([((g[:, 2] + g[:, 0]) / 2 - (a[:, 2] + a[:, 0]) / 2) / aw,
                      ((g[:, 3] + g[:, 1]) / 2 - (a[:, 3] + a[:, 1]) / 2) / ah,
                      np.log(gw / aw), np.log(gh / ah)], 1)
    return t / np.asarray(std, np.float64)


def encode_bound(gt, box, std=(1.0, 1.0, 1.0, 1.0)):
    """Per-component bound of the fp32 encode (every operation correctly rounded, logf within 1 ulp in CUDA):
    centre offsets: the two centres and their difference carry u (|g1| + |g2|) + u (|a1| + |a2|) each before the
    division, which adds u of the quotient; log(w_g / w_a): the widths carry u |w| each, the quotient u, logf u of
    its value plus 2 ulp absolute.  Division by std: u of the result."""
    g, a = np.asarray(gt, np.float64), np.asarray(box, np.float64)
    aw, ah = np.abs(a[:, 2] - a[:, 0]), np.abs(a[:, 3] - a[:, 1])
    gw, gh = np.abs(g[:, 2] - g[:, 0]), np.abs(g[:, 3] - g[:, 1])
    t = np.abs(encode64(gt, box))
    with np.errstate(divide="ignore", invalid="ignore"):
        bx = 3 * U * (np.abs(g[:, 0]) + np.abs(g[:, 2]) + np.abs(a[:, 0]) + np.abs(a[:, 2])) / aw + 3 * U * t[:, 0]
        by = 3 * U * (np.abs(g[:, 1]) + np.abs(g[:, 3]) + np.abs(a[:, 1]) + np.abs(a[:, 3])) / ah + 3 * U * t[:, 1]
        bw = 3 * U * ((np.abs(g[:, 0]) + np.abs(g[:, 2])) / gw + (np.abs(a[:, 0]) + np.abs(a[:, 2])) / aw) + 2 * U * t[:, 2] + 4 * U
        bh = 3 * U * ((np.abs(g[:, 1]) + np.abs(g[:, 3])) / gh + (np.abs(a[:, 1]) + np.abs(a[:, 3])) / ah) + 2 * U * t[:, 3] + 4 * U
    b = np.stack([bx, by, bw, bh], 1)
    return (b + 2 * U * t) / np.asarray(std, np.float64) + TINY


def check_encode(got, gt, box, std=(1.0, 1.0, 1.0, 1.0), what="encode"):
    """Finite components within the float64 bound; infinite ones (zero-width GT: log 0) equal the float64 value."""
    ref = encode64(gt, box, std)
    got = np.asarray(got)
    fin = np.isfinite(ref)
    assert np.array_equal(got[~fin], ref[~fin].astype(f32)) or (np.isnan(got[~fin]) == np.isnan(ref[~fin])).all(), what
    return within(got[fin], ref[fin], encode_bound(gt, box, std)[fin], what)


# ------------------------------------------------------------------------------------------------
# IoU constructions (find_jaccard_overlap in fp32: inter / (((area_a + area_b) - inter) + eps))
# ------------------------------------------------------------------------------------------------
def iou32(a, b, eps=1e-5):
    """Vectorised over a [..., 4] (fp32 operations in the kernel's order, b one box)."""
    a, b = np.asarray(a, f32), np.asarray(b, f32)
    w = np.maximum(np.minimum(a[..., 2], b[2]) - np.maximum(a[..., 0], b[0]), f32(0))
    h = np.maximum(np.minimum(a[..., 3], b[3]) - np.maximum(a[..., 1], b[1]), f32(0))
    inter = w * h
    aa = (a[..., 2] - a[..., 0]) * (a[..., 3] - a[..., 1])
    ab = (b[2] - b[0]) * (b[3] - b[1])
    return inter / (((aa + ab) - inter) + f32(eps))


def _ulps(x, k):
    """The 2k + 1 consecutive fp32 values centred on x."""
    i = np.asarray(x, f32).view(np.int32) + np.arange(-k, k + 1, dtype=np.int32)
    return i.view(f32)


@functools.lru_cache(maxsize=None)
def threshold_pair(target, side, eps=1e-5, gts=((0.25, 0.25, 0.75, 0.75), (0.1, 0.2, 0.7, 0.65))):
    """(anchor, GT): the anchor's fp32 IoU with the GT is exactly fp32(target) (side 0), or the fp32 IoU closest to
    it strictly below (side -1) / above (side +1) -- one ulp away where the search finds one (every case but just
    below 0.5f, where the quotient's ulp halves and the closest found is a few ulp away).  The anchor shares the GT's
    left and top edges; its right and bottom edges are searched over consecutive fp32 values around the real-valued
    solution, for the first GT of ``gts`` that has an exact hit."""
    tgt = f32(target)
    want = np.nextafter(tgt, f32(side * np.inf)) if side else tgt
    best = None
    for gt in gts:
        gt = np.asarray(gt, f32)
        w, h = float(gt[2] - gt[0]), float(gt[3] - gt[1])
        r = float(target) * (1 + 1e-5 / (w * h))              # anchor = GT shrunk in x to a fraction r of its width
        x2 = f32(gt[0] + r * w)
        xs, ys = _ulps(x2, 3000), _ulps(gt[3], 60)
        cand = np.zeros((len(ys), len(xs), 4), f32)
        cand[..., 0], cand[..., 1] = gt[0], gt[1]
        cand[..., 2], cand[..., 3] = xs[None, :], ys[:, None]
        iou = iou32(cand, gt, eps)
        hit = np.argwhere(iou == want)
        if len(hit):
            return cand[tuple(hit[0])], gt
        if side:
            ok = (iou < tgt) if side < 0 else (iou > tgt)
            dist = np.where(ok, np.abs(iou.astype(np.float64) - float(tgt)), np.inf)
            k = np.unravel_index(np.argmin(dist), dist.shape)
            if np.isfinite(dist[k]) and (best is None or dist[k] < best[0]):
                best = (dist[k], cand[k], gt)
    if best is None:
        raise AssertionError(f"no fp32 box within the search windows has IoU {want!r}")
    return best[1], best[2]


def slab_tie_case(N, S, variant="vgg"):
    """Caller-given anchors for one image of N anchors cut into S slabs as the RPN assign kernel cuts them (slabs of
    ceil(ceil(N / 32) / S) 32-anchor chunks): GT r - 1 (r = 1 .. S-1) is the dyadic square [r/8 - 1/8, r/8]^2 and its
    two best anchors are its left and right halves, placed at the last anchor of slab r - 1 and the first of slab r.
    All coordinates are dyadic, so both IoUs are computed exactly and tie bit for bit.  The other anchors are small
    boxes in [0.9, 0.99]^2 that overlap no GT.  Returns (anchors [N,4], gt [S-1,4], [(lo, hi) per GT])."""
    rs = np.random.RandomState(N + S)
    xy = rs.uniform(0.9, 0.98, (N, 2)).astype(f32)
    anchors = np.concatenate([xy, xy + f32(0.01)], 1).astype(f32)
    cpc = -(-(-(-N // 32)) // S)
    gts, ties = [], []
    for r in range(1, S):
        hi = r * cpc * 32
        if hi >= N:
            break
        x0 = f32((r - 1) / 8)
        gts.append([x0, x0, x0 + f32(0.125), x0 + f32(0.125)])
        anchors[hi - 1] = [x0, x0, x0 + f32(0.0625), x0 + f32(0.125)]
        anchors[hi] = [x0 + f32(0.0625), x0, x0 + f32(0.125), x0 + f32(0.125)]
        ties.append((hi - 1, hi))
    return anchors, np.asarray(gts, f32).reshape(-1, 4), ties
