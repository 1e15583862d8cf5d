"""CPU, only where the reference sources are available (oracle/ref_import.py): the oracle against the live, unmodified
reference."""
import os

import numpy as np
import pytest
import torch

from objectdetection_ssd_b200 import synth
from oracle import ref_import
from oracle import ssd_oracle as O

pytestmark = pytest.mark.skipif(not ref_import.available(), reason="unmodified reference sources not available (SSD_REFERENCE_DIR)")


def test_loss_grads_and_maps_bit_identical():
    RU, RL = ref_import.load()
    pri = O.make_priors()
    pxy = O.cxcywh_to_xyxy(pri)
    assert torch.equal(pri, RL.ancs_xywh) and torch.equal(pxy, RL.ancs_xyxy)
    B = 4
    gb, gc = synth.make_gt(11, B)
    loc, conf = synth.make_head(11, B, 8732)
    tb = [torch.from_numpy(b) for b in gb]
    tc = [torch.from_numpy(c) for c in gc]
    l = torch.from_numpy(loc).requires_grad_(True)
    c = torch.from_numpy(conf).requires_grad_(True)
    with ref_import.quiet():
        l1, l2 = RL.ssd((l, c), tc, tb)
        (l1 + l2).backward()
    r = O.multibox_loss(torch.from_numpy(loc), torch.from_numpy(conf), tb, tc, pri, pxy)
    assert r["loc_loss"].item() == l1.item() and r["conf_loss"].item() == l2.item()
    assert torch.equal(RL.obj_forEach_prior___.long(), r["cls"])
    gl, gcf = O.multibox_grads(torch.from_numpy(loc), torch.from_numpy(conf), r)
    assert torch.equal(gl, l.grad)
    assert torch.allclose(gcf, c.grad, rtol=1e-5, atol=1e-9)
    assert torch.equal(c.grad.abs().sum(-1) != 0, r["pos"] | r["mined"])
    # the reference-style op sequence (CPU baseline of bench.py) is the same computation bit for bit
    l_ = torch.from_numpy(loc).requires_grad_(True)
    c_ = torch.from_numpy(conf).requires_grad_(True)
    a, b = O.ssd_reference_style((l_, c_), tc, tb, pri, pxy)
    (a + b).backward()
    assert a.item() == l1.item() and b.item() == l2.item()
    assert torch.equal(l_.grad, l.grad) and torch.equal(c_.grad, c.grad)
    # legacy per-image variant
    with ref_import.quiet():
        o1, o2 = RL.ssd_old((torch.from_numpy(loc), torch.from_numpy(conf)), tc, tb)
    p1, p2 = O.ssd_per_image_mean((torch.from_numpy(loc), torch.from_numpy(conf)), tc, tb, pri, pxy)
    assert abs(o1.item() - p1.item()) < 1e-6 and abs(o2.item() - p2.item()) < 1e-5


def test_box_functions_bit_identical():
    RU, RL = ref_import.load()
    pri = O.make_priors()
    g = torch.randn(8732, 4, generator=torch.Generator().manual_seed(3))
    assert torch.equal(RU.gcxgcy_to_cxcy(g, pri), O.decode(g, pri))
    bx = O.cxcywh_to_xyxy(pri)
    assert torch.equal(RU.xyxy_to_xywh(bx), O.xyxy_to_cxcywh(bx))
    assert torch.equal(RU.get_offsets_coords(O.xyxy_to_cxcywh(bx)[:300], pri[100:400]),
                       O.encode(O.xyxy_to_cxcywh(bx)[:300], pri[100:400]))
    a = torch.rand(7, 4, generator=torch.Generator().manual_seed(4))
    a[:, 2:] = a[:, :2] + a[:, 2:] * 0.3
    assert torch.equal(RU.get_jaccard_tensor1(a, bx), O.iou_matrix(a, bx))


def test_detect_bit_identical():
    RU, RL = ref_import.load()
    pri = O.make_priors()
    dl, dc = synth.make_head(13, 1, 8732, loc_scale=0.5, bg_bias=8.5)
    with ref_import.quiet():
        bx, cl, pr = RL.inference(torch.from_numpy(dl[0]), torch.from_numpy(dc[0]), 0, toDraw=False,
                                  min_score=0.01, iou_threshold=0.45)
    b, c, p, _ = O.detect_image(torch.from_numpy(dl[0]), torch.from_numpy(dc[0]), pri, 0.01, 0.45, 200)
    assert torch.equal(bx, b) and torch.equal(cl, c) and torch.equal(pr, p)
    # nothing above threshold -> the reference returns three empty lists
    z = torch.zeros(8732, 21)
    z[:, 20] = 30.
    with ref_import.quiet():
        assert RL.inference(torch.from_numpy(dl[0]), z, 0, toDraw=False) == ([], [], [])
    assert O.detect_image(torch.from_numpy(dl[0]), z, pri)[0].shape[0] == 0


def test_frozen_fixture_holds_the_reference_values():
    """tests/golden/parity_golden.npz (what tests/test_parity_golden.py compares with) against the live reference."""
    from tests.golden.make_parity_golden import frozen_values
    G = np.load(os.path.join(os.path.dirname(__file__), "golden", "parity_golden.npz"), allow_pickle=False)
    want = frozen_values(live=True)
    assert set(want) <= set(G.files)
    for k, v in want.items():
        if k == "loss_old" or k.startswith("sgd_"):     # ssd_per_image_mean is pinned to 1e-6 / 1e-5, the loop to fp32
            assert np.allclose(G[k], v, rtol=1e-5, atol=1e-6), k
        else:
            assert np.array_equal(G[k], v), k
