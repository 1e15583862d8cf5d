"""The comparisons of tests/test_oracle_vs_reference.py against the frozen reference values of
tests/golden/parity_golden.npz (tests/golden/make_parity_golden.py), so that they run in every checkout: the oracle on
the CPU, the drop-in ssd() on the GPU."""
import os

import numpy as np
import pytest
import torch

from oracle import ssd_oracle as O
from tests.golden.make_parity_golden import box_inputs, detect_inputs, loss_inputs

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "parity_golden.npz"), allow_pickle=False)


def close(a, b, rtol=1e-6, atol=0.0):
    """Integer decisions are compared exactly; values that pass through exp / log / reductions only to fp32 rounding,
    which may differ between CPUs (vectorised transcendental functions)."""
    return a.shape == b.shape and np.allclose(a, b, rtol=rtol, atol=atol)


def test_box_functions_equal_the_frozen_reference():
    pri, g, bx, a = box_inputs()
    assert close(O.decode(g, pri).numpy(), G["box_decode"])
    assert np.array_equal(O.xyxy_to_cxcywh(bx).numpy(), G["box_cxcywh"])
    assert close(O.encode(O.xyxy_to_cxcywh(bx)[:300], pri[100:400]).numpy(), G["box_encode"], atol=1e-6)
    assert np.array_equal(O.iou_matrix(a, bx).numpy(), G["box_iou"])


def test_loss_grads_and_maps_equal_the_frozen_reference():
    pri = O.make_priors()
    pxy = O.cxcywh_to_xyxy(pri)
    loc, conf, tb, tc = loss_inputs()
    r = O.multibox_loss(loc, conf, tb, tc, pri, pxy)
    assert np.array_equal(r["cls"].numpy().astype(np.uint8), G["loss_cls"])
    assert close(np.array([r["loc_loss"].item(), r["conf_loss"].item()], np.float32), G["loss_losses"])
    gl, gcf = O.multibox_grads(loc, conf, r)
    assert close(gl.numpy(), G["loss_grad_loc"], 1e-5, 1e-9)
    assert close(gcf.numpy(), G["loss_grad_conf"], 1e-5, 1e-9)
    assert np.array_equal(np.abs(G["loss_grad_conf"]).sum(-1) != 0, (r["pos"] | r["mined"]).numpy())
    # the reference-style op sequence (CPU baseline of bench.py)
    l_ = loc.clone().requires_grad_(True)
    c_ = conf.clone().requires_grad_(True)
    a, b = O.ssd_reference_style((l_, c_), tc, tb, pri, pxy)
    (a + b).backward()
    assert close(np.array([a.item(), b.item()], np.float32), G["loss_losses"])
    assert close(l_.grad.numpy(), G["loss_grad_loc"], 1e-5, 1e-9) and close(c_.grad.numpy(), G["loss_grad_conf"], 1e-5, 1e-9)
    # legacy per-image variant (ssd_old)
    p1, p2 = O.ssd_per_image_mean((loc, conf), tc, tb, pri, pxy)
    assert abs(p1.item() - G["loss_old"][0]) < 1e-6 and abs(p2.item() - G["loss_old"][1]) < 1e-5


def test_detect_equals_the_frozen_reference():
    pri = O.make_priors()
    dl, dc = detect_inputs()
    b, c, p, _ = O.detect_image(dl, dc, pri, 0.01, 0.45, 200)
    assert b.shape[0] > 0
    assert np.array_equal(c.numpy().astype(np.int32), G["detect_cls"])
    assert close(b.numpy(), G["detect_boxes"], atol=1e-6) and close(p.numpy(), G["detect_prob"])
    z = torch.zeros(8732, 21)          # nothing above threshold: the reference returns three empty lists
    z[:, 20] = 30.
    assert O.detect_image(dl, z, pri)[0].shape[0] == 0


def test_voc_ap_equals_the_frozen_reference_get_map():
    from tests.test_evalmap import MAP_CASES, synth_eval
    for i, (seed, images) in enumerate(MAP_CASES):
        assert np.array_equal(O.voc_ap(*synth_eval(seed, images)), G["map_ap"][i])


@pytest.mark.gpu
def test_dropin_ssd_equals_the_frozen_reference():
    from objectdetection_ssd_b200 import Losses
    loc, conf, tb, tc = loss_inputs()
    l = loc.cuda().requires_grad_(True)
    c = conf.cuda().requires_grad_(True)
    l1, l2 = Losses.ssd((l, c), tc, tb)
    (l1 + l2).backward()
    assert close(np.array([l1.item(), l2.item()], np.float32), G["loss_losses"], 1e-5)
    assert close(l.grad.cpu().numpy(), G["loss_grad_loc"], 1e-5, 1e-9)
    assert close(c.grad.cpu().numpy(), G["loss_grad_conf"], 1e-5, 1e-9)
