"""The fused region loss (frr_region_loss through ops.region_loss and torch.ops.frr.region_loss) against a float64
reference written in tests/training_refs.py, independent of oracle/: every loss component and every gradient element
within a written fp32 error bound, at the shapes, launch geometries and edges the kernel accepts; NaN / inf where the
reference's own fp32 torch expression gives them; and the kernel's bitwise invariants (batch independence, run-to-run
reproducibility, gathered == ungathered class rows, requested-gradient subsets, the total's summation order)."""
import itertools

import numpy as np
import pytest
import torch

import training_refs as tr
from faster_rcnn_pytorch_b200 import _lib, ops, torch_ops  # noqa: F401  (registers torch.ops.frr)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
f32 = np.float32
KNOTS_RPN = [tr.RPN_BETA, -tr.RPN_BETA, np.nextafter(tr.RPN_BETA, f32(0)), np.nextafter(tr.RPN_BETA, f32(1)),
             f32(1.0), -f32(1.0), np.nextafter(f32(1), f32(0)), np.nextafter(f32(1), f32(2)), f32(0.0)]
KNOTS_FRC = [f32(1.0), -f32(1.0), np.nextafter(f32(1), f32(0)), np.nextafter(f32(1), f32(2)),
             tr.RPN_BETA, -np.nextafter(tr.RPN_BETA, f32(0)), f32(0.0), -f32(0.0)]


def dev(a, grad=False):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t.requires_grad_(True) if grad else t


def make_image(seed, N, S, C, CR, n_pos, n_neg, frc_pos, pad=None, knots=True):
    """One image: ``N`` anchors with n_pos positives and n_neg negatives at random places, ``S`` Fast R-CNN rows with
    frc_pos foreground rows (class C-1 among them), the rows in ``pad`` marked as padding; the first positives of both
    halves carry SmoothL1 differences exactly on and one ulp around the knots (beta, 1) and exactly 0."""
    rs = np.random.RandomState(seed)
    x = {}
    if N:
        t = np.full(N, -1, np.int64)
        sel = rs.permutation(N)[:n_pos + n_neg]
        t[sel[:n_pos]], t[sel[n_pos:]] = 1, 0
        rr = (rs.standard_normal((N, 4)) * 0.3).astype(f32)
        rtr = (rs.standard_normal((N, 4)) * 0.3).astype(f32)
        if knots:
            for j, i in enumerate(np.sort(sel[:n_pos])[:len(KNOTS_RPN)]):
                rtr[i] = 0.0
                rr[i] = [KNOTS_RPN[(j + k) % len(KNOTS_RPN)] for k in range(4)]
        x.update(rpn_cls=(rs.standard_normal((N, 2)) * 2).astype(f32), rpn_reg=rr, rpn_tcls=t, rpn_treg=rtr)
    if S:
        c = np.zeros(S, np.int64)
        if C > 1 and frc_pos:
            c[:frc_pos] = rs.randint(1, C, frc_pos)
            c[0] = C - 1
        if pad is not None:
            c[pad] = -1
        fr = rs.standard_normal((S, CR, 4)).astype(f32)
        ftr = rs.standard_normal((S, 4)).astype(f32)
        if knots:
            for j, s in enumerate(np.nonzero(c > 0)[0][:len(KNOTS_FRC)]):
                ftr[s] = 0.0
                fr[s, 0 if CR == 1 else c[s]] = [KNOTS_FRC[(j + k) % len(KNOTS_FRC)] for k in range(4)]
        x.update(frc_cls=(rs.standard_normal((S, C)) * 2).astype(f32), frc_reg=fr, frc_tcls=c, frc_treg=ftr)
    return x


def stack(xs, key):
    return None if xs[0].get(key) is None else np.stack([x[key] for x in xs])


def run(xs, g=None, via="ops"):
    """The kernel on a batch: loss [B,5] and the gradients of sum(loss * g) (g [B,5], default: the totals)."""
    B = len(xs)
    keys = ("rpn_cls", "rpn_reg", "frc_cls", "frc_reg")
    preds = {k: (None if xs[0].get(k) is None else dev(stack(xs, k), True)) for k in keys}
    tg = {k: (None if xs[0].get(k) is None else dev(stack(xs, k))) for k in ("rpn_tcls", "rpn_treg", "frc_tcls", "frc_treg")}
    args = (preds["rpn_cls"], preds["rpn_reg"], tg["rpn_tcls"], tg["rpn_treg"], preds["frc_cls"], preds["frc_reg"],
            tg["frc_tcls"], tg["frc_treg"])
    loss = ops.region_loss(*args) if via == "ops" else torch.ops.frr.region_loss(*args)[0]
    gg = torch.zeros((B, 5), device=DEV) if g is None else dev(np.asarray(g, f32))
    if g is None:
        gg[:, 0] = 1
    (loss * gg).sum().backward()
    grads = [None if preds[k] is None else preds[k].grad.cpu().numpy() for k in keys]
    return loss.detach().cpu().numpy(), grads


def check_batch(xs, loss, grads, g=None, check_grads=True):
    worst = np.zeros(5)
    for b, x in enumerate(xs):
        ref = tr.loss_reference(x, None if g is None else g[b])
        worst = np.maximum(worst, tr.check_loss(loss[b], ref, f"image {b} loss"))
        if not check_grads or not ref["finite"].all():
            continue
        for j, name in enumerate(("rpn_cls", "rpn_reg", "frc_cls", "frc_reg")):
            if ref["grads"][j] is None:
                continue
            got = grads[j][b].reshape(ref["grads"][j].shape)
            tr.within(got, ref["grads"][j], ref["gbound"][j], f"image {b} d/d{name}")
    return worst


# B, N, S, C, frcnn_reg_rows ("C" or 1), halves, n_pos, n_neg, frc_pos
SHAPES = [
    (1, 1, 1, 1, "C", "both", 1, 0, 0),
    (3, 31, 31, 2, "C", "both", 5, 26, 9),
    (3, 1024, 32, 21, "C", "both", 100, 924, 10),
    (3, 1025, 33, 31, 1, "both", 300, 725, 33),
    (1, 20646, 128, 21, "C", "both", 40, 216, 32),
    (3, 37350, 512, 81, "C", "both", 128, 128, 128),
    (1, 267069, 1100, 91, "C", "both", 3000, 50000, 300),
    (64, 20646, 128, 21, 1, "both", 40, 216, 32),
    (3, 20646, 128, 32, "C", "rpn", 256, 0, 0),
    (3, 0, 33, 33, "C", "frc", 0, 0, 33),
    (1, 0, 1100, 1024, "C", "frc", 0, 0, 700),
    (2, 1025, 1, 1024, 1, "both", 1025, 0, 1),
    (3, 1024, 512, 91, "C", "frc", 0, 0, 0),
]


@pytest.mark.parametrize("B,N,S,C,CR,halves,n_pos,n_neg,frc_pos", SHAPES,
                         ids=[f"B{s[0]}-N{s[1]}-S{s[2]}-C{s[3]}-R{s[4]}-{s[5]}" for s in SHAPES])
def test_region_loss_shapes_vs_float64(B, N, S, C, CR, halves, n_pos, n_neg, frc_pos):
    cr = C if CR == "C" else 1
    xs = []
    for b in range(B):
        pad = np.arange(1, S, 3) if (b % 2 and S > 2) else None          # padding rows interleaved with real ones
        x = make_image(1000 * B + b, N if halves != "frc" else 0, S if halves != "rpn" else 0, C, cr, n_pos, n_neg,
                       frc_pos, pad)
        xs.append(x)
    loss, grads = run(xs)
    check_batch(xs, loss, grads)
    # rows outside the sample get exactly zero gradient
    if halves != "frc":
        t = stack(xs, "rpn_tcls")
        assert not grads[0][t < 0].any() and not grads[1][t <= 0].any()
    if halves != "rpn":
        c = stack(xs, "frc_tcls")
        assert not grads[2][c < 0].any() and not grads[3][c <= 0].any()


def test_region_loss_bound_catches_one_missing_term_and_a_normaliser_off_by_one():
    """The bound is tight enough for the changes it must see at N = 20 646 with 256 sampled anchors (~4e-3 relative)."""
    x = make_image(77, 20646, 128, 21, 21, 40, 216, 32)
    loss, _ = run([x])
    ref = tr.loss_reference(x)
    tr.check_loss(loss[0], ref)
    for q, n in ((1, 256), (3, 128)):
        off = ref["loss"][q] * n / (n + 1)
        assert abs(off - ref["loss"][q]) > 20 * ref["bound"][q], (q, ref["bound"][q])


EDGES = ["rpn_all_ignored", "frc_all_padding", "no_positives", "all_positive", "interleaved_padding", "class_C_minus_1",
         "knots_only"]


@pytest.mark.parametrize("edge", EDGES)
def test_region_loss_target_edges(edge):
    N, S, C = 4100, 128, 21
    x = make_image(60 + EDGES.index(edge), N, S, C, C, 30, 200, 32)
    if edge == "rpn_all_ignored":
        x["rpn_tcls"][:] = -1                       # nv = 0: both RPN losses NaN (0 / 0 like the reference), no gradient
    elif edge == "frc_all_padding":
        x["frc_tcls"][:] = -1
    elif edge == "no_positives":
        x["rpn_tcls"][x["rpn_tcls"] > 0] = 0
        x["frc_tcls"][:] = 0
    elif edge == "all_positive":
        x["rpn_tcls"][x["rpn_tcls"] == 0] = 1
        x["frc_tcls"][:] = np.random.RandomState(5).randint(1, C, S)
    elif edge == "interleaved_padding":
        x["frc_tcls"][1::2] = -1
    elif edge == "class_C_minus_1":
        x["frc_tcls"][:64] = C - 1
    elif edge == "knots_only":                      # every positive difference on a knot: the sums are exact
        x["rpn_tcls"][:] = -1
        x["rpn_tcls"][:9] = 1
        x["rpn_treg"][:9] = 0
        x["rpn_reg"][:9] = np.asarray([[KNOTS_RPN[(j + k) % 9] for k in range(4)] for j in range(9)], f32)
    g = np.asarray([[1.0, -0.5, 2.0, 0.0, 3.0]], f32)
    loss, grads = run([x], g)
    ref = tr.loss_reference(x, g[0])
    tr.check_loss(loss[0], ref)
    if edge == "rpn_all_ignored":
        assert np.isnan(loss[0, :3]).all() and not grads[0].any() and not grads[1].any()
    elif edge == "frc_all_padding":
        assert np.isnan(loss[0, [0, 3, 4]]).all() and not grads[2].any() and not grads[3].any()
    elif edge == "no_positives":
        assert loss[0, 2] == 0 and loss[0, 4] == 0 and not grads[1].any() and not grads[3].any()
    else:
        check_batch([x], loss, grads, g)
    if edge == "knots_only":
        # |d| >= beta is linear: |d| - beta / 2; below it 0.5 d^2 / beta -- both exact in fp32 at these differences
        b = tr.RPN_BETA
        d = np.abs(x["rpn_reg"][:9])
        terms = np.where(d >= b, d - f32(0.5) * b, f32(0.5) * d * d / b).astype(np.float64)
        assert float(loss[0, 2]) == pytest.approx(terms.sum() / 9, rel=4 * 40 * tr.U)


@pytest.mark.parametrize("beta", [0.05, 0.054918307811021805, 1.4527008533477783])
def test_smooth_l1_branch_exactly_at_beta(monkeypatch, beta):
    """A difference exactly on beta takes the linear branch (|d| >= beta).  At the project's betas (fp32(1/9), 1) both
    branches round to the same fp32 value there, so the ABI is driven with betas where they do not."""
    b = f32(beta)
    lin, quad = f32(b - f32(0.5) * b), f32(f32(f32(0.5) * b) * b) / b
    assert lin != quad, "this beta does not separate the two branches"
    monkeypatch.setattr(ops, "RPN_BETA", float(b))
    monkeypatch.setattr(ops, "FRCNN_BETA", float(b))
    x = make_image(3, 64, 8, 5, 5, 1, 3, 1, knots=False)
    p = np.nonzero(x["rpn_tcls"] > 0)[0][0]
    x["rpn_treg"][p] = 0
    x["rpn_reg"][p] = [b, 0, 0, 0]                  # one term on the knot, three exactly 0: the sums are exact
    x["frc_treg"][0] = 0
    x["frc_reg"][0, x["frc_tcls"][0]] = [0, -b, 0, 0]
    loss, grads = run([x])
    assert loss[0, 2] == lin / f32(4) and loss[0, 4] == lin / f32(8)        # 4 sampled anchors, 8 rows
    ref = tr.loss_reference(x, rpn_beta=b, frcnn_beta=b)
    tr.check_loss(loss[0], ref)
    assert np.array_equal(grads[1][0, p], np.asarray([1, 0, 0, 0], f32) / f32(4))
    assert np.array_equal(grads[3][0, 0, x["frc_tcls"][0]], np.asarray([0, -1, 0, 0], f32) / f32(8))


EXTREMES = ["pm1e4", "equal", "neg_inf_other", "neg_inf_target", "pos_inf", "all_neg_inf", "fltmax"]


@pytest.mark.parametrize("where", ["rpn", "frc"])
@pytest.mark.parametrize("kind", EXTREMES)
def test_region_loss_extreme_logits(kind, where):
    """Finite results within the float64 bound; NaN / inf exactly where the reference's fp32 torch cross entropy gives
    them (+inf in a logit: NaN; -inf in the target class: +inf; -inf elsewhere: finite)."""
    C = 33
    x = make_image(11, 2000, 64, C, C, 20, 100, 16)
    key, tkey = ("rpn_cls", "rpn_tcls") if where == "rpn" else ("frc_cls", "frc_tcls")
    l, t = x[key], x[tkey]
    rows = np.nonzero(t >= 0)[0][:6]
    for r in rows:
        tc = int(t[r])
        other = (tc + 1) % l.shape[1]
        if kind == "pm1e4":
            l[r] = np.where(np.arange(l.shape[1]) % 2, 1e4, -1e4)
        elif kind == "equal":
            l[r] = 3.5
        elif kind == "neg_inf_other":
            l[r, other] = -np.inf
        elif kind == "neg_inf_target":
            l[r, tc] = -np.inf
        elif kind == "pos_inf":
            l[r, other] = np.inf
        elif kind == "all_neg_inf":
            l[r] = -np.inf
        elif kind == "fltmax":
            l[r, tc], l[r, other] = np.finfo(f32).max, -np.finfo(f32).max
    loss, grads = run([x])
    ref = tr.loss_reference(x)
    tr.check_loss(loss[0], ref)
    if kind in ("pm1e4", "equal", "neg_inf_other", "fltmax"):
        assert np.isfinite(loss[0]).all()
        check_batch([x], loss, grads)
    elif kind == "neg_inf_target":
        assert loss[0, 1 if where == "rpn" else 3] == np.inf
    else:
        assert np.isnan(loss[0, 1 if where == "rpn" else 3])


@pytest.mark.parametrize("via", ["ops", "torch_ops"])
def test_region_loss_gradients_with_upstream_weights(via):
    """Upstream g [B,5] with zeros, negatives and per-component weights, through both front ends."""
    xs = [make_image(500 + b, 5000, 128, 21, 21, 20 + b, 200, 10 + b, np.arange(90, 128) if b == 2 else None)
          for b in range(4)]
    g = np.asarray([[0, 2, 0, 0, 0], [1, 0, 0, 0, 3], [0, 0, 0, 1, 0], [-1.5, 0.25, -2, 4, 0.5]], f32)
    loss, grads = run(xs, g, via)
    check_batch(xs, loss, grads, g)
    assert not grads[1][0].any() and grads[0][0].any()
    assert not grads[0][2].any() and not grads[3][2].any() and grads[2][2].any()


def test_region_loss_class_at_or_above_C_counts_in_normaliser_only():
    """A Fast R-CNN class >= C is not checked on the host (that would synchronise a captured / compiled step): it counts
    in the normaliser and adds no loss term and no gradient (documented with frr_region_loss in include/frr.h)."""
    C = 21
    x = make_image(8, 1000, 64, C, C, 10, 50, 20)
    x["frc_tcls"][[3, 7]] = [C, C + 40]
    loss, grads = run([x])
    ref = tr.loss_reference(x)
    tr.check_loss(loss[0], ref)
    assert not grads[2][0, [3, 7]].any() and not grads[3][0, [3, 7]].any()
    y = {k: v.copy() for k, v in x.items()}
    y["frc_tcls"][[3, 7]] = -1                        # padding instead: one term fewer in the normaliser, same sums
    ly, _ = run([y])
    assert ly[0, 3] * 62 == pytest.approx(loss[0, 3] * 64, rel=1e-6)


# ------------------------------------------------------------------------------------------------ bitwise invariants
def _kernel(xs, need=(True,) * 4):
    args = ops.region_loss_args(*[None if stack(xs, k) is None else dev(stack(xs, k)) for k in
                                  ("rpn_cls", "rpn_reg", "rpn_tcls", "rpn_treg", "frc_cls", "frc_reg", "frc_tcls", "frc_treg")])
    loss, grads = ops.region_loss_kernel(*args, need=need)
    return loss.cpu().numpy(), [None if g is None else g.cpu().numpy() for g in grads]


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def test_region_loss_bitwise_invariants():
    xs = [make_image(900 + b, 20646, 128, 21, 21, 40 + b % 7, 216, 8 + b % 20, np.arange(100, 128) if b % 5 == 0 else None)
          for b in range(65)]
    loss, grads = _kernel(xs)
    # two runs, identical bits
    loss2, grads2 = _kernel(xs)
    assert np.array_equal(_bits(loss), _bits(loss2))
    for a, b in zip(grads, grads2):
        assert np.array_equal(_bits(a), _bits(b))
    # each image alone == the same image inside the batch of 65
    for b in (0, 1, 31, 64):
        lb, gb = _kernel(xs[b:b + 1])
        assert np.array_equal(_bits(lb[0]), _bits(loss[b]))
        for a, full in zip(gb, grads):
            assert np.array_equal(_bits(a[0]), _bits(full[b]))
    # the total is ((rpn_cls + rpn_reg) + frcnn_cls) + frcnn_reg in fp32
    t = torch.from_numpy(loss)
    tot = ((t[:, 1] + t[:, 2]) + t[:, 3]) + t[:, 4]
    assert np.array_equal(_bits(tot.numpy()), _bits(loss[:, 0]))
    # every subset of requested gradients: the same bits for the ones requested, the loss unchanged
    small = xs[:3]
    lf, gf = _kernel(small)
    for need in itertools.product((False, True), repeat=4):
        ln, gn = _kernel(small, need)
        assert np.array_equal(_bits(ln), _bits(lf)), need
        for j in range(4):
            assert (gn[j] is None) == (not need[j])
            if need[j]:
                assert np.array_equal(_bits(gn[j]), _bits(gf[j])), (need, j)


@pytest.mark.parametrize("C", [1, 2, 21, 33, 81])
def test_region_loss_gathered_rows_equal_class_rows(C):
    """frcnn_reg_rows = 1 on the rows gathered at the target class == frcnn_reg_rows = C, bit for bit."""
    xs = [make_image(40 + b, 1025, 130, C, C, 30, 300, 40, np.arange(0, 130, 4) if b else None) for b in range(3)]
    lf, gf = _kernel(xs)
    gath = []
    for x in xs:
        y = dict(x)
        c = np.maximum(x["frc_tcls"], 0)
        y["frc_reg"] = x["frc_reg"][np.arange(len(c)), c][:, None, :].copy()
        gath.append(y)
    lg, gg = _kernel(gath)
    assert np.array_equal(_bits(lf), _bits(lg))
    for b, x in enumerate(xs):
        c = np.maximum(x["frc_tcls"], 0)
        assert np.array_equal(_bits(gf[3][b][np.arange(len(c)), c]), _bits(gg[3][b][:, 0]))
    assert np.array_equal(_bits(gf[2]), _bits(gg[2]))


def test_region_loss_launches_one_kernel():
    x = make_image(1, 1025, 33, 21, 21, 10, 100, 5)
    before = _lib.launch_count()
    _kernel([x])
    assert _lib.launch_count() - before == 1


@pytest.fixture(scope="module", autouse=True)
def _report_worst_ratios():
    yield
    print("\nworst error/bound ratios (loss):", {k: round(v, 4) for k, v in sorted(tr.WORST.items())})
