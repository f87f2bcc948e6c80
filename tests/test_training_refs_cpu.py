"""CPU self-checks of the references in tests/training_refs.py that the GPU tests of the region loss and the target
makers rely on: the threshold pairs and slab ties are what they claim to be in fp32, the float64 loss reference agrees
with the oracle on the golden loss inputs, and the bound helpers accept the reference and reject a perturbed copy."""
import numpy as np
import pytest

import training_refs as tr
from faster_rcnn_pytorch_b200 import synth
from conftest import golden
from oracle import region_oracle

f32 = np.float32


@pytest.mark.parametrize("target", [0.7, 0.3, 0.5])
def test_threshold_pairs_hit_the_fp32_thresholds(target):
    t = f32(target)
    box, gt = tr.threshold_pair(target, 0)
    assert tr.iou32(box, gt) == t
    assert region_oracle.pairwise_iou_eps(box[None], gt[None])[0, 0] == t        # the oracle's IoU is the same fp32 value
    below, gb = tr.threshold_pair(target, -1)
    above, ga = tr.threshold_pair(target, +1)
    lo, hi = tr.iou32(below, gb), tr.iou32(above, ga)
    assert lo < t < hi
    assert hi == np.nextafter(t, f32(1))
    ulps = int(t.view(np.int32)) - int(f32(lo).view(np.int32))
    assert 1 <= ulps <= (2 if target == 0.5 else 1), ulps


def test_slab_ties_are_bitwise_ties():
    for variant in ("vgg", "fpn"):
        anchors, gt, ties = tr.slab_tie_case(20646, 8, variant)
        eps = 1e-5 if variant == "vgg" else 0.0
        iou = region_oracle.pairwise_iou_eps(anchors, gt, eps)
        for g, (lo, hi) in enumerate(ties):
            col = iou[:, g]
            assert col[lo].view(np.uint32) == col[hi].view(np.uint32)
            assert col[lo] == col.max() and col[lo] > 0
            assert np.count_nonzero(col == col.max()) == 2
            assert hi == lo + 1


@pytest.mark.parametrize("name,kw", [("voc", dict(seed=8300, N=20646, S=128, C=21)),
                                     ("coco", dict(seed=8301, N=37350, S=128, C=81, n_pos=128, n_neg=128))])
def test_float64_loss_reference_matches_oracle_on_golden_inputs(name, kw):
    x = synth.loss_inputs(**kw)
    ref = tr.loss_reference(x)
    want = region_oracle.region_loss(x["rpn_cls"], x["rpn_reg"], x["rpn_tcls"], x["rpn_treg"], x["frc_cls"], x["frc_reg"],
                                      x["frc_tcls"], x["frc_treg"])
    np.testing.assert_allclose(ref["loss"], want, rtol=1e-6)
    np.testing.assert_allclose(ref["loss"], golden("loss")[f"{name}_loss"], rtol=1e-5)


def test_bound_helpers_accept_the_reference_and_reject_a_perturbed_copy():
    x = synth.loss_inputs(seed=8300, N=20646, S=128, C=21)
    ref = tr.loss_reference(x)
    tr.check_loss(ref["loss"].astype(f32), ref)                         # the reference rounded to fp32 passes
    for q in range(1, 5):
        bad = ref["loss"].copy()
        bad[q] *= 256 / 257                                              # a normaliser off by one
        with pytest.raises(AssertionError):
            tr.check_loss(bad, ref)
    for j in range(4):
        gr = ref["grads"][j]
        tr.within(gr.astype(f32), gr, ref["gbound"][j], "self")
        nz = np.argwhere(gr != 0)[0]
        bad = gr.copy()
        bad[tuple(nz)] *= 1 + 1e-4
        with pytest.raises(AssertionError):
            tr.within(bad, gr, ref["gbound"][j], "perturbed")
    gt = synth.gt_boxes(1, 6)[0]
    box = synth.random_boxes(2, 6)[0]
    enc = tr.encode64(gt, box)
    tr.check_encode(enc.astype(f32), gt, box)
    with pytest.raises(AssertionError):
        tr.check_encode((enc * (1 + 1e-5)).astype(f32), gt, box)
