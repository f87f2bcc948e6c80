"""GPU: the detection tail -- decode_classwise (D1), class_nms (D2) and both evaluation packers -- against plain
references written here, independent of oracle/, at the shapes and edges the entry points accept:

  * D1 numerics vs float64 torch on the CPU; under extreme head outputs (logits of +-1e4 and -inf, t.z = +-500,
    rois of zero width or height) NaN, +-inf, 0 and 1 sit exactly where the reference's own fp32 torch expression
    (models/model.py:369-378) puts them;
  * D2 bit for bit vs torchvision.ops.nms on the CPU, per image and class, on the kernel's own fp32 inputs: R from 1 to
    4096 (every bitonic sort size), C from 2 to 1024, B up to 64, ragged and clamped roi counts, thresholds that select
    the screened and the exact keep-list kernel, disjoint / identical / flat / exact-threshold boxes, score ties, caps;
  * the class-major and the score-ranked packers vs a stable torch sort, including a cap above 65 536;
  * argument checks that refuse before anything is launched.
"""
import math

import numpy as np
import pytest
import torch
import torchvision

from faster_rcnn_pytorch_b200 import _lib, ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
STD = torch.tensor([0.1, 0.1, 0.2, 0.2], dtype=torch.float32)  # the fp32 constants of models/model.py:372
NAN = float("nan")


def dev(a):
    return torch.as_tensor(np.ascontiguousarray(a)).to(DEV)


def bits(t):
    return t.contiguous().view(torch.int32)


# ------------------------------------------------------------------------------------------------ D1 references
def decode_ref64(cls, reg, rois):
    """float64: softmax of the fp32 logits, reg * the fp32 std, decode against the roi's centre and size, corners,
    clamp to [0, 1]."""
    C = cls.shape[1]
    prob = torch.softmax(cls.double(), dim=1)
    t = reg.double().reshape(-1, C, 4) * STD.double()
    r = rois.double().reshape(-1, 1, 4)
    rw, rh = r[..., 2] - r[..., 0], r[..., 3] - r[..., 1]
    cx, cy = t[..., 0] * rw + (r[..., 0] + r[..., 2]) / 2, t[..., 1] * rh + (r[..., 1] + r[..., 3]) / 2
    w, h = torch.exp(t[..., 2]) * rw, torch.exp(t[..., 3]) * rh
    b = torch.stack([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], dim=-1).clamp(0, 1)
    return prob, b.reshape(-1, C * 4)


def decode_ref32(cls, reg, rois):
    """The reference's fp32 expression (models/model.py:369-378 with utils/util.py xy_to_cxcy / decode / cxcy_to_xy):
    the one that decides where inf and NaN appear (exp(88.8) overflows in fp32, not in float64)."""
    C = cls.shape[1]
    prob = torch.softmax(cls, dim=-1)
    t = (reg.reshape(-1, C, 4) * STD).reshape(-1, 4)
    r = rois.reshape(-1, 1, 4).expand(-1, C, 4).reshape(-1, 4)
    rc = torch.cat([(r[:, 2:] + r[:, :2]) / 2, r[:, 2:] - r[:, :2]], 1)
    d = torch.cat([t[:, :2] * rc[:, 2:] + rc[:, :2], torch.exp(t[:, 2:]) * rc[:, 2:]], 1)
    xy = torch.cat([d[:, :2] - d[:, 2:] / 2, d[:, :2] + d[:, 2:] / 2], 1)
    return prob, xy.reshape(-1, C * 4).clamp(min=0, max=1)


def head_inputs(seed, rows, C, scale=1.0):
    cls, reg = synth.head_outputs(seed, rows, C)
    rois = synth.random_boxes(seed + 1, max(rows, 1))[0][:rows]
    return torch.from_numpy(cls * np.float32(scale)), torch.from_numpy(reg), torch.from_numpy(rois)


def extreme_inputs(seed, rows, C):
    """Head outputs at the edges of fp32: logits of +-1e4, rows with -inf logits and row 3 all -inf; t.z / t.w of
    +-500 and 443 / 444 (0.2 * t just below / above the fp32 overflow of exp); rois of zero width, height or both."""
    cls, reg, rois = head_inputs(seed, rows, C)
    cls, reg, rois = cls.clone(), reg.clone().reshape(rows, C, 4), rois.clone()
    for r in range(rows):
        kind = r % 6
        if kind == 0:
            cls[r, r % C] = 1e4
        elif kind == 1:
            cls[r, r % C] = -1e4
        elif kind == 2:
            cls[r, ::2] = -math.inf
        elif kind == 4:
            cls[r, ::2], cls[r, 1::2] = 1e4, -1e4
        if r % 5 == 0:
            rois[r, 2] = rois[r, 0]
        elif r % 5 == 1:
            rois[r, 3] = rois[r, 1]
        elif r % 5 == 2:
            rois[r, 2:] = rois[r, :2]
    cls[3] = -math.inf
    big = torch.tensor([500.0, -500.0, 443.0, 444.0, 0.5])
    reg[:, :, 2] = big[torch.arange(rows * C).reshape(rows, C) % 5]
    reg[:, :, 3] = big[(torch.arange(rows * C).reshape(rows, C) + 2) % 5]
    return cls, reg.reshape(rows, C * 4), rois


def run_decode(cls, reg, rois, C):
    prob, boxes = ops.decode_classwise(dev(cls), dev(reg), dev(rois), C)
    return prob.cpu(), boxes.cpu()


@pytest.mark.parametrize("rows,C", [(0, 21), (1, 21), (7, 2), (8, 33), (9, 1), (300, 2), (300, 31), (300, 32),
                                    (300, 33), (64, 1024), (1000, 81), (2000, 91)])
def test_decode_classwise_vs_float64(rows, C):
    """rows 0 / 1 / 7 / 8 / 9 around the 8 rows of a CTA; C around the 32 lanes of the warp that owns a row.  Tighter
    than the stated contract (prob rtol 1e-5 / atol 1e-7, boxes rtol 1e-5 / atol 1e-6): on a B200 (1000 W limit) the
    errors at these shapes stay below 0.12 (prob) and 0.38 (boxes) of the bounds used here."""
    cls, reg, rois = head_inputs(1000 + rows + C, rows, C, scale=3.0)
    prob, boxes = run_decode(cls, reg, rois, C)
    assert prob.shape == (rows, C) and boxes.shape == (rows, 4 * C)
    wp, wb = decode_ref64(cls, reg, rois)
    torch.testing.assert_close(prob.double(), wp, rtol=2e-6, atol=1e-7)
    torch.testing.assert_close(boxes.double(), wb, rtol=1e-5, atol=2e-7)


def special_masks(t):
    return {"nan": t.isnan(), "+inf": t.isposinf(), "-inf": t.isneginf(), "0": t == 0, "1": t == 1}


@pytest.mark.parametrize("rows,C", [(7, 2), (8, 21), (9, 33), (300, 81)])
def test_decode_classwise_extremes(rows, C):
    """NaN / +-inf / 0 / 1 exactly where the reference's fp32 expression has them (a roi of zero width with
    exp(0.2 t.z) = inf gives inf * 0 = NaN there, and clamp keeps NaN); every other value within the float64 tolerance."""
    cls, reg, rois = extreme_inputs(2000 + rows, rows, C)
    prob, boxes = run_decode(cls, reg, rois, C)
    rp, rb = decode_ref32(cls, reg, rois)
    for what, got, want in (("prob", prob, rp), ("boxes", boxes, rb)):
        gm, wm = special_masks(got), special_masks(want)
        for k in gm:
            bad = (gm[k] != wm[k]).nonzero()
            assert bad.numel() == 0, f"{what}: '{k}' differs at {bad[:8].tolist()}"
    assert rb.isnan().any() and rp[3].isnan().all()      # the edges were reached
    wp, wb = decode_ref64(cls, reg, rois)
    wb[rb.isnan()] = NAN
    torch.testing.assert_close(prob.double(), wp, rtol=1e-5, atol=1e-7, equal_nan=True)
    torch.testing.assert_close(boxes.double(), wb, rtol=1e-5, atol=1e-6, equal_nan=True)


# ------------------------------------------------------------------------------------------------ D2
def class_nms_ref(prob, boxes, thres, iou_thr, roi_count, cap):
    """FRCNN._suppress per image on the CPU with torchvision.ops.nms (stable descending sort, fp32 IoU compared in
    double): rows prob[:, l] > thres for every class l >= 1, concatenated class-major with label l - 1, first cap rows.
    prob [B,R,C], boxes [B,R,C,4] fp32."""
    B, R, C = prob.shape
    out = []
    for b in range(B):
        n = R if roi_count is None else max(0, min(int(roi_count[b]), R))
        bl, ll, sl = [], [], []
        for l in range(1, C):
            s = prob[b, :n, l]
            m = s > thres
            bx, sc = boxes[b, :n, l][m], s[m]
            k = torchvision.ops.nms(bx, sc, iou_thr)
            bl.append(bx[k])
            sl.append(sc[k])
            ll.append(torch.full((len(k),), l - 1, dtype=torch.int32))
        out.append((torch.cat(bl)[:cap], torch.cat(ll)[:cap], torch.cat(sl)[:cap]))
    return out


def assert_det_equal(det, ref):
    db, dl, ds, dc = (t.cpu() for t in det)
    assert dc.shape == (len(ref),)
    for b, (rb, rl, rs) in enumerate(ref):
        n = len(rl)
        assert int(dc[b]) == n, f"image {b}: count {int(dc[b])} != {n}"
        assert torch.equal(dl[b, :n], rl), f"image {b}: labels differ"
        assert torch.equal(bits(ds[b, :n]), bits(rs)), f"image {b}: scores differ"
        assert torch.equal(bits(db[b, :n]), bits(rb)), f"image {b}: boxes differ"
        assert (dl[b, n:] == -1).all() and (bits(ds[b, n:]) == 0).all() and (bits(db[b, n:]) == 0).all()


def quantised_prob(rs, B, R, C):
    """Softmax probabilities rounded to k/64: many exact ties inside and across classes."""
    x = rs.standard_normal((B, R, C)) * 2
    p = np.exp(x) / np.exp(x).sum(-1, keepdims=True)
    return (np.round(p * 64) / 64).astype(np.float32)


def grid_boxes(rs, R, C):
    """Per class a permutation of R boxes, each inset in its own cell of a grid: pairwise disjoint, so every box is
    kept at any threshold and the kept list spans R / 256 chunks."""
    side = math.ceil(math.sqrt(R))
    i = np.arange(R)
    x0, y0 = (i % side) / side, (i // side) / side
    cell = np.stack([x0 + 0.1 / side, y0 + 0.1 / side, x0 + 0.9 / side, y0 + 0.9 / side], 1)
    return np.stack([cell[rs.permutation(R)] for _ in range(C)], 1).astype(np.float32)


def flat_boxes(rs, R, C):
    """Random boxes, every third one clamped flat against the right border (x1 = x2 = 1) and every third one against the
    top (y1 = y2 = 0), as decode produces for boxes outside the image."""
    b = synth.random_boxes(int(rs.randint(1 << 30)), R * C)[0].reshape(R, C, 4)
    b[0::3, :, 0] = b[0::3, :, 2] = 1.0
    b[1::3, :, 1] = b[1::3, :, 3] = 0.0
    return b


# IoU of the nested boxes [0, y, a, y + 1] and [0, y, b, y + 1] is b / a exactly: fp32(thr) itself
EXACT_IOU = {0.0: (0, 10), 1e-7: (1, 10 ** 7), 0.3: (3, 10), 0.5: (5, 10), 0.7: (7, 10), 1.0: (10, 10)}


def exact_iou_boxes(thr, R, C):
    """Pairs of nested boxes whose IoU is fl32(thr), one numerator unit below or above it, stacked along y with gaps."""
    num, den = EXACT_IOU[thr]
    assert np.float32(num) / np.float32(den) == np.float32(thr)
    i = np.arange(R)
    g = i // 2
    x2 = np.where(i % 2 == 0, den, np.clip(num + (g % 3) - 1, 0, None)).astype(np.float64)
    b = np.stack([np.zeros(R), 2.0 * g, x2, 2.0 * g + 1], 1)
    return np.repeat(b[:, None], C, 1).astype(np.float32)


def detection_inputs(kind, seed, B, R, C, iou_thr=0.3):
    """prob [B,R,C], boxes [B,R,C*4] on the device."""
    rs = np.random.RandomState(seed)
    if kind in ("decode", "decode_extreme"):
        mk = (lambda: head_inputs(seed, B * R, C, scale=3.0)) if kind == "decode" else (lambda: extreme_inputs(seed, B * R, C))
        cls, reg, rois = mk()
        prob, boxes = ops.decode_classwise(dev(cls), dev(reg), dev(rois), C)
        return prob.reshape(B, R, C), boxes.reshape(B, R, C * 4)
    if kind in ("random", "ties"):
        prob = quantised_prob(rs, B, R, C) if kind == "random" else np.full((B, R, C), 0.25, np.float32)
        boxes = np.stack([synth.random_boxes(seed + 1 + b, R * C)[0] for b in range(B)])
    elif kind == "grid":
        prob = rs.uniform(0.06, 1.0, (B, R, C)).astype(np.float32)
        boxes = np.stack([grid_boxes(rs, R, C) for _ in range(B)])
    elif kind == "identical":                             # one box per class, all scores equal
        prob = np.full((B, R, C), 0.25, np.float32)
        boxes = np.broadcast_to(synth.random_boxes(seed, B * C)[0].reshape(B, 1, C, 4), (B, R, C, 4))
    elif kind == "flat":
        prob = quantised_prob(rs, B, R, C)
        boxes = np.stack([flat_boxes(rs, R, C) for _ in range(B)])
    elif kind == "exact_iou":
        prob = quantised_prob(rs, B, R, C)
        boxes = np.broadcast_to(exact_iou_boxes(iou_thr, R, C), (B, R, C, 4))
    else:
        raise AssertionError(kind)
    return dev(prob), dev(np.reshape(boxes, (B, R, C * 4)))


def roi_counts(kind, B, R):
    if kind is None:
        return None
    if kind == "ragged":                                  # full, none, and values in between
        v = [R, 0] + [int(x) for x in np.random.RandomState(R).randint(1, R + 1, max(B - 2, 0))]
        return np.asarray(v[:B] if B > 1 else [R // 2 + 1], np.int32)
    if kind == "over":                                    # above R: the kernel clamps to R
        return np.asarray([R + 1, 2 ** 31 - 1, 4 * R][:B], np.int32)
    return np.full(B, {"zero": 0, "one": 1, "full": R}[kind], np.int32)


def expected_variant(iou_thr):
    """The keep-list kernel screens pairs without a division only for finite thresholds >= 1e-6."""
    return "screened" if math.isfinite(iou_thr) and iou_thr >= 1e-6 else "exact"


def check_class_nms(prob, boxes, B, R, C, thres, iou_thr, rc=None, cap=None):
    v = ops.nms_variant(B * (C - 1), R, iou_thr, R, cluster_size=1, threads=256)
    assert (v["variant"], v["cluster_size"], v["threads"]) == (expected_variant(iou_thr), 1, 256)
    det = ops.class_nms(prob, boxes, C, score_thres=thres, iou_thr=iou_thr, roi_count=None if rc is None else dev(rc),
                        cap=cap)
    full = R * (C - 1) if cap is None else cap
    assert det[1].shape == (B, full)
    ref = class_nms_ref(prob.cpu(), boxes.cpu().reshape(B, R, C, 4), thres, iou_thr, rc, full)
    assert_det_equal(det, ref)
    return det, ref, v


D2_CASES = [
    # B, R, C, inputs, roi_count, score_thres, iou_thr
    (3, 1, 21, "decode", None, 0.05, 0.3),
    (1, 31, 33, "random", "ragged", 3 / 64, 0.5),          # threshold equal to quantised scores: > is not >=
    (3, 32, 1024, "decode", "full", 0.0, 0.3),             # C - 1 = 1023 classes: the compaction's prefix at its limit
    (3, 33, 91, "decode", "over", 0.005, 0.7),
    (3, 255, 2, "flat", "ragged", 0.05, 0.3),
    (1, 256, 21, "grid", None, 0.05, 0.0),                 # exact kernel, kept list of exactly one chunk
    (3, 257, 21, "grid", "ragged", 0.05, 1e-7),            # exact kernel, one candidate into the second chunk
    (64, 300, 81, "decode", "ragged", 0.05, 0.3),          # the infer batch shape
    (3, 300, 21, "random", "one", 0.0, 0.3),
    (2, 300, 21, "random", "zero", 0.05, 0.3),
    (3, 300, 21, "ties", "ragged", 0.05, 0.5),             # every score equal: stable order is the row order
    (2, 300, 81, "decode_extreme", None, 0.05, 0.3),       # NaN boxes from decode never suppress and are never suppressed
    (1, 64, 1024, "random", "full", 0.0, 0.5),
    (1, 1000, 81, "decode", None, 0.05, 0.5),              # FPN test-mode proposals, torchvision box-head threshold
    (3, 1023, 3, "identical", None, 0.05, 1.0),            # IoU 1 is not > 1: every row kept, 4 chunks
    (1, 1024, 3, "identical", "over", 0.05, 0.3),          # one row kept per class
    (3, 1025, 2, "flat", "ragged", 0.5, 0.7),
    (1, 2000, 21, "decode", None, 0.0, 0.7),
    (1, 4096, 3, "grid", None, 0.05, 0.3),                 # > 4000 kept per class: a 4097-box slice (> 48 KB)
    (1, 4096, 2, "grid", "full", 0.05, NAN),               # exact kernel, nothing suppressed
]


@pytest.mark.parametrize("B,R,C,kind,roi,thres,iou_thr", D2_CASES,
                         ids=[f"B{c[0]}-R{c[1]}-C{c[2]}-{c[3]}-roi_{c[4]}-s{c[5]:.4g}-iou{c[6]}" for c in D2_CASES])
def test_class_nms_vs_torchvision(B, R, C, kind, roi, thres, iou_thr):
    prob, boxes = detection_inputs(kind, 3000 + R + C, B, R, C)
    det, ref, v = check_class_nms(prob, boxes, B, R, C, thres, iou_thr, roi_counts(roi, B, R))
    if R == 4096:
        assert v["smem"] > 48 * 1024
    if kind == "grid" and R == 4096:
        assert int(det[3][0]) > 4000 * (C - 1)


@pytest.mark.parametrize("iou_thr", sorted(EXACT_IOU))
def test_class_nms_iou_equal_to_threshold(iou_thr):
    """IoU == fl32(thr) is suppressed exactly when fl32(thr) > thr in double (0.3, 1e-7), kept otherwise (0, 0.5, 0.7,
    1): the keep lists of torchvision's CPU kernel."""
    B, R, C = 3, 300, 21
    prob, boxes = detection_inputs("exact_iou", 3500, B, R, C, iou_thr)
    _, ref, _ = check_class_nms(prob, boxes, B, R, C, 0.0, iou_thr)
    # below 1 both decisions occur among the pairs; at 1 nothing is suppressed
    n, kept = int((prob.cpu()[:, :, 1:] > 0).sum()), sum(len(r[1]) for r in ref)
    assert (0 < kept < n) if iou_thr < 1 else kept == n


@pytest.mark.parametrize("cap_kind", ["0", "1", "total-1", "total", "default"])
def test_class_nms_cap(cap_kind):
    """The first cap class-major rows of every image and count = min(total, cap); cap = 0 asks for the counts alone.
    Both packers take the truncated rows as they are."""
    B, R, C = 3, 300, 21
    prob, boxes = detection_inputs("random", 3600, B, R, C)
    rc = roi_counts("ragged", B, R)
    total = max(len(r[1]) for r in class_nms_ref(prob.cpu(), boxes.cpu().reshape(B, R, C, 4), 0.05, 0.3, rc, R * C))
    cap = {"0": 0, "1": 1, "total-1": total - 1, "total": total, "default": None}[cap_kind]
    det, _, _ = check_class_nms(prob, boxes, B, R, C, 0.05, 0.3, rc, cap)
    check_pack(det, 100, "class", 0, use_wh=True, xywh=True)
    check_pack(det, 100, "score", 1, use_wh=False, xywh=False)


# ------------------------------------------------------------------------------------------------ evaluation hand-off
def pack_ref(db, dl, ds, dc, max_det, rank, per_class_max, wh, xywh):
    """[B,max_det,6] rows (x, y, x2|w, y2|h, score, label) and counts: rank="class" takes the first max_det rows,
    rank="score" a stable descending sort of the rows that are among the first per_class_max of their class."""
    B, cap = dl.shape
    out = torch.zeros((B, max_det, 6), dtype=torch.float32)
    cnt = torch.zeros(B, dtype=torch.int32)
    for b in range(B):
        n = max(0, min(int(dc[b]), cap))
        rows = torch.arange(n)
        if rank == "score":
            if per_class_max > 0:
                lab = dl[b, :n]
                order = torch.sort(lab, stable=True).indices
                sl = lab[order]
                start = torch.ones(n, dtype=torch.bool)
                start[1:] = sl[1:] != sl[:-1]
                first = torch.cummax(torch.where(start, torch.arange(n), 0), 0).values if n else rows
                in_class = torch.empty(n, dtype=torch.int64)
                in_class[order] = torch.arange(n) - first
                rows = rows[in_class < per_class_max]
            rows = rows[torch.sort(ds[b, rows], descending=True, stable=True).indices]
        rows = rows[:max_det]
        k = len(rows)
        s = torch.ones(2) if wh is None else wh[b]
        bx = db[b, rows] * torch.stack([s[0], s[1], s[0], s[1]])
        if xywh:
            bx = torch.cat([bx[:, :2], bx[:, 2:] - bx[:, :2]], 1)
        out[b, :k] = torch.cat([bx, ds[b, rows, None], dl[b, rows, None].float()], 1)
        cnt[b] = k
    return out, cnt


_DETS = {}


def ranked_det(shape):
    """Detections of class_nms, built once per module: 'b3_r300_c81' (ragged, tied scores: cap 24 000) and
    'b1_r1000_c81' (cap 79 920 > 65 536: the general radix top-k with a validity mask)."""
    if shape not in _DETS:
        if shape == "b3_r300_c81":
            prob, boxes = detection_inputs("random", 3700, 3, 300, 81)
            _DETS[shape] = ops.class_nms(prob, boxes, 81, score_thres=0.005, iou_thr=0.5, roi_count=dev(np.int32([300, 120, 0])))
        else:
            prob, boxes = detection_inputs("decode", 3701, 1, 1000, 81)
            _DETS[shape] = ops.class_nms(prob, boxes, 81, score_thres=0.0, iou_thr=0.5)
    return _DETS[shape]


WH = torch.tensor([[1333.0, 800.0], [640.0, 480.0], [500.0, 375.0]])


def check_pack(det, max_det, rank, per_class_max, use_wh, xywh):
    B = det[1].shape[0]
    wh = WH[:B] if use_wh else None
    got, gc = ops.pack_detections(*det, max_det, image_wh=None if wh is None else dev(wh), xywh=xywh, rank=rank,
                                  per_class_max=per_class_max)
    want, wc = pack_ref(*(t.cpu() for t in det), max_det, rank, per_class_max, wh, xywh)
    assert torch.equal(gc.cpu(), wc)
    assert torch.equal(bits(got.cpu()), bits(want))


@pytest.mark.parametrize("shape", ["b3_r300_c81", "b1_r1000_c81"])
@pytest.mark.parametrize("max_det", [1, 100, 16384])
@pytest.mark.parametrize("per_class_max", [0, 1, 100])
def test_pack_ranked_vs_stable_sort(shape, max_det, per_class_max):
    det = ranked_det(shape)
    if shape == "b1_r1000_c81":
        assert det[1].shape[1] > 65536 and int(det[3][0]) > 16384
    check_pack(det, max_det, "score", per_class_max, use_wh=max_det != 100, xywh=per_class_max == 1)


@pytest.mark.parametrize("shape", ["b3_r300_c81", "b1_r1000_c81"])
@pytest.mark.parametrize("max_det", [1, 100, 16384])
def test_pack_class_major_vs_reference(shape, max_det):
    check_pack(ranked_det(shape), max_det, "class", 0, use_wh=max_det == 100, xywh=max_det == 1)


# ------------------------------------------------------------------------------------------------ argument edges
def test_argument_checks_launch_nothing():
    """class_nms refuses R > 4096, C > 1024 and C < 2 (a class list needs a background class), and the ranked packer a
    workspace that is too small, before any kernel is launched.  decode_classwise accepts C = 1 (tested above)."""
    bad = [(4097, 2), (1, 1025), (1, 1)]
    ins = [(torch.zeros((1, R, C), device=DEV), torch.zeros((1, R, 4 * C), device=DEV)) for R, C in bad]
    det = (torch.zeros((2, 8, 4), device=DEV), torch.zeros((2, 8), dtype=torch.int32, device=DEV),
           torch.zeros((2, 8), device=DEV), torch.full((2,), 8, dtype=torch.int32, device=DEV))
    small = torch.empty(16, dtype=torch.uint8, device=DEV)
    torch.cuda.synchronize()
    before = _lib.launch_count()
    for (R, C), (prob, boxes) in zip(bad, ins):
        with pytest.raises(ValueError, match="frr_class_nms"):
            ops.class_nms(prob, boxes, C)
    with pytest.raises(_lib.FrrError, match=r"failed \(-3\).*workspace too small"):
        ops.pack_detections(*det, 4, rank="score", workspace=small)
    assert _lib.launch_count() == before
