"""GPU parity: the per-pyramid-level entry points (SURVEY.md 8(f) #3) against the concatenated ones - the same kernels
reading the level tensors in place, so every result must be bit-identical - and against the oracle."""
import pytest
import torch

from oracle import ssd_oracle as O
from tests import helpers as H

pytestmark = pytest.mark.gpu

SSD300_LEVELS = (5776, 2166, 600, 150, 36, 4)


def _head(pri):
    from objectdetection_ssd_b200.head import MultiboxHead
    return MultiboxHead(pri, "cuda")


def _split(t, counts):
    out, s = [], 0
    for n in counts:
        out.append(t[:, s:s + n].contiguous())
        s += n
    return out


@pytest.mark.parametrize("B", [3, 32, 256, 300])
def test_loss_levels_equals_concatenated(B):
    """B = 300 is more images than the 2 CTAs x 148 SMs of a B200 the mining kernel can hold co-resident: both routes
    take the separate finaliser and the ordinary mining kernel (three launches instead of two)."""
    from objectdetection_ssd_b200 import _lib
    from objectdetection_ssd_b200.head import PackedGT
    pri = H.priors()
    loc, conf, tb, tc = H.train_inputs(51, B, pri.shape[0])
    head = _head(pri)
    gt = PackedGT(tb, tc, head.dev)
    ref = head.loss(loc.cuda(), conf.cuda(), gt, with_grads=True)
    loc_lv, conf_lv = _split(loc.cuda(), SSD300_LEVELS), _split(conf.cuda(), SSD300_LEVELS)
    n0 = _lib.launch_count()
    lv = head.loss_levels(loc_lv, conf_lv, gt, with_grads=True)
    launches = _lib.launch_count() - n0
    torch.cuda.synchronize()
    if B >= 256:
        coresident = 2 * torch.cuda.get_device_properties(0).multi_processor_count   # 2 mining CTAs per SM
        assert launches == (3 if B > coresident else 2), launches
    assert torch.equal(lv["losses"], ref["losses"]) and torch.equal(lv["sums"], ref["sums"])
    assert torch.equal(lv["npos"], ref["npos"]) and torch.equal(lv["cls_u8"], ref["cls_u8"])
    assert torch.equal(lv["best_prior"], ref["best_prior"])
    assert torch.equal(torch.cat(lv["grad_loc"], 1), ref["grad_loc"])
    assert torch.equal(torch.cat(lv["grad_conf"], 1), ref["grad_conf"])


def test_loss_levels_against_the_oracle_and_autograd():
    from objectdetection_ssd_b200 import Losses
    pri = H.priors()
    B = 8
    loc, conf, tb, tc = H.train_inputs(52, B, pri.shape[0])
    locs = [t.cuda().requires_grad_(True) for t in _split(loc, SSD300_LEVELS)]
    confs = [t.cuda().requires_grad_(True) for t in _split(conf, SSD300_LEVELS)]
    l1, l2 = Losses.ssd_levels((locs, confs), [c.cuda() for c in tc], [b.cuda() for b in tb])
    (2.0 * l1 + 0.5 * l2).backward()
    lo, co = loc.clone().requires_grad_(True), conf.clone().requires_grad_(True)
    r1, r2 = O.ssd_reference_style((lo, co), tc, tb, pri, O.cxcywh_to_xyxy(pri))
    (2.0 * r1 + 0.5 * r2).backward()
    assert torch.allclose(l1.cpu(), r1.detach(), rtol=1e-5) and torch.allclose(l2.cpu(), r2.detach(), rtol=1e-5)
    gl = torch.cat([t.grad for t in locs], 1).cpu()
    gc = torch.cat([t.grad for t in confs], 1).cpu()
    assert torch.allclose(gl, lo.grad, rtol=1e-5, atol=1e-9)
    assert torch.allclose(gc, co.grad, rtol=1e-4, atol=1e-8)


def test_loss_levels_forward_only_and_bad_level_sum():
    from objectdetection_ssd_b200.head import PackedGT
    pri = H.priors()
    loc, conf, tb, tc = H.train_inputs(53, 4, pri.shape[0])
    head = _head(pri)
    gt = PackedGT(tb, tc, head.dev)
    ref = head.loss(loc.cuda(), conf.cuda(), gt, with_grads=False)
    lv = head.loss_levels(_split(loc.cuda(), SSD300_LEVELS), _split(conf.cuda(), SSD300_LEVELS), gt, with_grads=False)
    assert torch.equal(lv["losses"], ref["losses"])
    with pytest.raises(ValueError):
        head.loss_levels(_split(loc.cuda(), SSD300_LEVELS)[:5], _split(conf.cuda(), SSD300_LEVELS)[:5], gt, with_grads=False)


def test_loss_levels_from_nhwc_conv_maps():
    """The real thing: channels_last conv outputs, permute is a view, no copy before the kernels."""
    from objectdetection_ssd_b200 import Losses
    from objectdetection_ssd_b200.head import PackedGT
    pri = H.priors()
    B = 2
    loc, conf, tb, tc = H.train_inputs(54, B, pri.shape[0])
    grids = ((38, 4), (19, 6), (10, 6), (5, 6), (3, 4), (1, 4))
    loc_maps, conf_maps, s = [], [], 0
    for hw, a in grids:
        n = hw * hw * a
        lm = loc[:, s:s + n].reshape(B, hw, hw, a * 4).permute(0, 3, 1, 2)          # NCHW view of NHWC memory
        cm = conf[:, s:s + n].reshape(B, hw, hw, a * 21).permute(0, 3, 1, 2)
        loc_maps.append(lm.cuda().contiguous(memory_format=torch.channels_last))
        conf_maps.append(cm.cuda().contiguous(memory_format=torch.channels_last))
        s += n
    locs, confs = Losses.head_levels(loc_maps, conf_maps)
    assert all(t.is_contiguous() for t in locs + confs)                              # views of the conv outputs
    assert locs[0].data_ptr() == loc_maps[0].data_ptr()
    head = _head(pri)
    gt = PackedGT(tb, tc, head.dev)
    ref = head.loss(loc.cuda(), conf.cuda(), gt, with_grads=True)
    lv = head.loss_levels(locs, confs, gt, with_grads=True)
    assert torch.equal(lv["losses"], ref["losses"])
    assert torch.equal(torch.cat(lv["grad_conf"], 1), ref["grad_conf"])


@pytest.mark.parametrize("bias,B", [(6.0, 3), (8.0, 64)])
def test_detect_levels_equals_concatenated(bias, B):
    from objectdetection_ssd_b200.head import detect, detect_levels
    pri = H.priors()
    loc, conf = H.detect_inputs(55, B, pri.shape[0], bg_bias=bias)
    head = _head(pri)
    ref = detect(head, loc.cuda(), conf.cuda(), 0.01, 0.45, 200)
    out = detect_levels(head, _split(loc.cuda(), SSD300_LEVELS), _split(conf.cuda(), SSD300_LEVELS), 0.01, 0.45, 200)
    torch.cuda.synchronize()
    assert torch.equal(out["cnt"], ref["cnt"])
    for i in range(B):
        k = int(ref["cnt"][i])
        for key in ("boxes", "prob", "cls", "prior"):
            assert torch.equal(out[key][i, :k], ref[key][i, :k]), (i, key)


def test_levels_random_splits_equal_concatenated():
    """Random level structures (1..8 levels, odd and tiny counts, rows not multiples of 4 -> plain-load tails): loss,
    gradients and detections must stay bit-identical to the concatenated calls."""
    from objectdetection_ssd_b200.head import PackedGT, detect, detect_levels
    g = torch.Generator().manual_seed(77)
    pri = H.priors()
    P = pri.shape[0]
    head = _head(pri)
    for trial in range(8):
        B = [1, 2, 5, 16][trial % 4]
        L = int(torch.randint(1, 9, (1,), generator=g))
        cuts = sorted(set(int(x) for x in torch.randint(1, P, (L - 1,), generator=g).tolist()))
        if trial == 3:
            cuts = [P - 7, P - 3, P - 2, P - 1]                  # tiny levels at the end: warps span many images
        if trial == 5:
            cuts = [1, 2, 5]                                     # ... and at the start
        counts = [b - a for a, b in zip([0] + cuts, cuts + [P])]
        loc, conf, tb, tc = H.train_inputs(60 + trial, B, P)
        gt = PackedGT(tb, tc, head.dev)
        ref = head.loss(loc.cuda(), conf.cuda(), gt, with_grads=True)
        lv = head.loss_levels(_split(loc.cuda(), counts), _split(conf.cuda(), counts), gt, with_grads=True)
        torch.cuda.synchronize()
        msg = f"trial {trial}: B={B} counts={counts}"
        assert torch.equal(lv["losses"], ref["losses"]) and torch.equal(lv["sums"], ref["sums"]), msg
        assert torch.equal(lv["cls_u8"], ref["cls_u8"]) and torch.equal(lv["best_prior"], ref["best_prior"]), msg
        assert torch.equal(torch.cat(lv["grad_loc"], 1), ref["grad_loc"]), msg
        assert torch.equal(torch.cat(lv["grad_conf"], 1), ref["grad_conf"]), msg
        dl, dc = H.detect_inputs(70 + trial, B, P, bg_bias=7.0)
        r = detect(head, dl.cuda(), dc.cuda(), 0.01, 0.45, 100)
        o = detect_levels(head, _split(dl.cuda(), counts), _split(dc.cuda(), counts), 0.01, 0.45, 100)
        torch.cuda.synchronize()
        assert torch.equal(o["cnt"], r["cnt"]), msg
        for i in range(B):
            k = int(r["cnt"][i])
            for key in ("boxes", "prob", "cls", "prior"):
                assert torch.equal(o[key][i, :k], r[key][i, :k]), (msg, i, key)
