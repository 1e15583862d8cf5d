"""GPU: the CUDA kernels against the FROZEN outputs of the unmodified reference (tests/golden/ssd_golden.npz, made by
tests/golden/make_golden.py from the reference sources) - directly, without the oracle in between, so that a regression of the
oracle cannot hide one of the kernels.  Integer / boolean results (class map, object map, positive counts, rows that
carry a gradient) are compared exactly; losses, gradient checksums, probabilities and boxes to 1e-5 relative (fp32)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from objectdetection_ssd_b200 import synth
from objectdetection_ssd_b200 import priors as PR

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ssd_golden.npz")


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def _head(pri):
    from objectdetection_ssd_b200.head import MultiboxHead
    return MultiboxHead(pri, "cuda")


def test_train_step_against_the_frozen_reference(gold):
    from objectdetection_ssd_b200.head import PackedGT
    B, P = 8, 8732
    pri = PR.make_priors()
    gb, gc = synth.make_gt(1, B)
    loc, conf = synth.make_head(1, B, P)
    assert synth.digest(loc, conf, *gb, *gc) == str(gold["train_digest"]), "inputs differ from the frozen run's"
    tb = [torch.from_numpy(b) for b in gb]
    tc = [torch.from_numpy(c) for c in gc]
    head = _head(pri)
    gt = PackedGT(tb, tc, head.dev)
    out = head.loss(torch.from_numpy(loc).cuda(), torch.from_numpy(conf).cuda(), gt, with_grads=True)
    torch.cuda.synchronize()
    losses = out["losses"].cpu().numpy()
    assert np.allclose(losses, gold["train_losses"], rtol=1e-5, atol=0), (losses, gold["train_losses"])
    # class map after the forced override (Losses.obj_forEach_prior___), positives per image: exact
    assert np.array_equal(out["cls_u8"].cpu().numpy(), gold["train_cls"])
    assert np.array_equal(out["npos"].cpu().numpy()[:B], gold["train_npos"])
    # object map (map_prior_to_bb, local gt index per prior, forced override included): exact, from the debug tap
    m = head.match(gt, want_maps=True)
    off = torch.tensor(gt.off_host[:-1]).view(B, 1)
    assert np.array_equal((m["obj"].cpu() - off).numpy().astype(np.int16), gold["train_obj_local"])
    # rows that carry a conf gradient = positives + mined negatives (T4)
    rows = (out["grad_conf"] != 0).any(-1).cpu().numpy()
    ref_rows = np.unpackbits(gold["train_grad_rows"], axis=1)[:, :P].astype(bool)
    if not np.array_equal(rows, ref_rows):
        # a flip is legitimate only AT the mining boundary: the CE of every differing row must sit within 4 ulp of the
        # smallest CE the reference mined in that image (torch fp32 CE as the yardstick)
        ce = F.cross_entropy(torch.from_numpy(conf).view(-1, 21), torch.from_numpy(gold["train_cls"]).view(-1).long(),
                             reduction="none").view(B, P).numpy()
        pos = gold["train_cls"] != 20
        for b in range(B):
            bad = np.nonzero(rows[b] != ref_rows[b])[0]
            if bad.size:
                edge = ce[b][ref_rows[b] & ~pos[b]].min()
                assert np.all(np.abs(ce[b][bad] - edge) <= 4 * np.spacing(np.float32(edge))), (b, bad, ce[b][bad], edge)
    else:
        gl, gcf = out["grad_loc"].cpu(), out["grad_conf"].cpu()
        got = np.array([gl.abs().sum().item(), gcf.abs().sum().item(), gl.sum().item(),
                        (gcf * torch.arange(21.)).sum().item()])
        assert np.allclose(got[:2], gold["train_grad_sums"][:2], rtol=1e-5)
        assert np.allclose(got[2:], gold["train_grad_sums"][2:], rtol=1e-3, atol=1e-4)      # signed sums cancel


def test_tie_rules_against_the_frozen_reference(gold):
    """T1-T3 on hand-made gts: identical boxes (last gt wins the forced prior), a degenerate box, repeated tiny boxes."""
    from objectdetection_ssd_b200.head import PackedGT
    pri = PR.make_priors()
    box = torch.tensor([[0.2, 0.2, 0.6, 0.7]])
    tb = [torch.cat([box, box, box]), torch.tensor([[0.5, 0.5, 0.5, 0.5], [0.1, 0.1, 0.3, 0.3]]),
          torch.tensor([[0.3, 0.3, 0.31, 0.31], [0.3, 0.3, 0.31, 0.31], [0.9, 0.9, 1.0, 1.0]])]
    tc = [torch.tensor([3., 7., 5.]), torch.tensor([1., 2.]), torch.tensor([0., 4., 8.])]
    head = _head(pri)
    gt = PackedGT(tb, tc, head.dev)
    m = head.match(gt, want_maps=True)
    torch.cuda.synchronize()
    off = torch.tensor(gt.off_host[:-1]).view(3, 1)
    assert np.array_equal(m["cls"].cpu().numpy().astype(np.uint8), gold["ties_cls"])
    assert np.array_equal((m["obj"].cpu() - off).numpy().astype(np.int16), gold["ties_obj"])


def test_fused_detect_against_the_frozen_reference(gold):
    """inference() of the reference at min_score 0.01 (more than top_k survive -> global score order): the fused
    kernels' detections, compared as (class, probability, box) records."""
    from objectdetection_ssd_b200.head import detect
    P = 8732
    pri = PR.make_priors()
    dl, dc = synth.make_head(3, 2, P, loc_scale=0.5, bg_bias=8.0)
    assert synth.digest(dl, dc) == str(gold["detect_digest"])
    out = detect(_head(pri), torch.from_numpy(dl), torch.from_numpy(dc), 0.01, 0.45, 200)
    torch.cuda.synchronize()
    for i in range(2):
        rb, rc, rp = gold[f"detect_boxes_{i}"], gold[f"detect_cls_{i}"], gold[f"detect_prob_{i}"]
        k = int(out["cnt"][i])
        assert k == rb.shape[0]
        gb, gcl, gp = out["boxes"][i, :k].cpu().numpy(), out["cls"][i, :k].cpu().numpy(), out["prob"][i, :k].cpu().numpy()
        assert np.all(np.diff(gp) <= 0), "more than top_k survive: descending score order (Losses.py:77-81)"
        used, unmatched = set(), 0
        for j in range(k):
            hit = [q for q in np.nonzero((rc == gcl[j]) & (np.abs(rp - gp[j]) <= 1e-5 * rp))[0]
                   if q not in used and np.allclose(rb[q], gb[j], rtol=1e-5, atol=1e-6)]
            if hit:
                used.add(hit[0])
            else:
                unmatched += 1
        # a record can only be missing at the top-k cut (two probabilities a few ulp apart swapping places)
        assert unmatched <= 1, f"image {i}: {unmatched} detections without a counterpart in the frozen reference output"
        if unmatched:
            assert abs(gp[-1] - rp[-1]) <= 1e-5 * rp[-1]


def test_stress_shape_against_the_frozen_reference(gold):
    from objectdetection_ssd_b200.head import PackedGT
    pri = PR.make_priors(PR.SSD512_SPEC)
    import hashlib
    assert hashlib.sha256(np.ascontiguousarray(pri.numpy()).tobytes()).hexdigest() == str(gold["stress_priors_sha"])
    gb, gc = synth.make_gt(5, 1, 100, 100)
    loc, conf = synth.make_head(5, 1, pri.shape[0])
    assert synth.digest(loc, conf, *gb, *gc) == str(gold["stress_digest"])
    head = _head(pri)
    gt = PackedGT([torch.from_numpy(b) for b in gb], [torch.from_numpy(c) for c in gc], head.dev)
    out = head.loss(torch.from_numpy(loc).cuda(), torch.from_numpy(conf).cuda(), gt, with_grads=False)
    torch.cuda.synchronize()
    assert np.allclose(out["losses"].cpu().numpy(), gold["stress_losses"], rtol=1e-5, atol=0)
    assert np.array_equal(out["cls_u8"].cpu().numpy(), gold["stress_cls"])
