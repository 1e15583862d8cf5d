"""GPU parity: decode + score threshold + per-class NMS + global top-k against the CPU oracle.

Stage-isolated (the oracle's decoded boxes and probabilities are fed to the kernels): keep lists, classes,
prior ids and order are bit-exact under T5-T7.  End to end (the kernels' own expf): decoded boxes and
probabilities agree to 1e-5 and the detections match except where a score or IoU sits within a few ulp of
its threshold, which the test accounts for explicitly.
"""
import pytest
import torch
import torch.nn.functional as F

from oracle import ssd_oracle as O
from tests import helpers as H

pytestmark = pytest.mark.gpu


def _head(pri):
    from objectdetection_ssd_b200.head import MultiboxHead
    return MultiboxHead(pri, "cuda")


def _oracle_stage(boxes, probs, min_score, iou_thr, top_k):
    return [O.detect_from_scores(boxes[i], probs[i], min_score, iou_thr, top_k) for i in range(boxes.shape[0])]


def _same_bits(a, b, signed_zero=True):
    """Bit-for-bit equality of two fp32 tensors, except that any NaN equals any NaN (payloads are not specified) and,
    with signed_zero=False, -0.0 equals +0.0 (a given score of -0.0 is reported as +0.0, see ssdhead.h)."""
    a, b = a.cpu(), b.cpu()
    if a.shape != b.shape:
        return False
    same = (a.view(torch.int32) == b.view(torch.int32)) | (torch.isnan(a) & torch.isnan(b))
    if not signed_zero:
        same |= (a == 0) & (b == 0)
    return bool(same.all())


def _check_exact(out, ref, top_k, what=""):
    cnt = out["cnt"].cpu()
    for i, (rb, rc, rp, ri) in enumerate(ref):
        k = int(cnt[i])
        assert k == rb.shape[0], f"{what} image {i}: {k} detections, oracle {rb.shape[0]}"
        assert torch.equal(out["prior"][i, :k].cpu().long(), ri), f"{what} image {i}: prior ids / order"
        assert torch.equal(out["cls"][i, :k].cpu().long(), rc), f"{what} image {i}: classes"
        assert _same_bits(out["prob"][i, :k], rp, signed_zero=False), f"{what} image {i}: scores"
        assert _same_bits(out["boxes"][i, :k], rb), f"{what} image {i}: boxes"


@pytest.mark.parametrize("bias,min_score,B", [(8.0, 0.01, 4), (6.0, 0.01, 2), (6.0, 0.2, 3), (2.0, 0.05, 2)])
def test_detect_from_scores_exact(bias, min_score, B):
    from objectdetection_ssd_b200.head import detect_from_scores
    pri = H.priors()
    loc, conf = H.detect_inputs(31, B, pri.shape[0], bg_bias=bias)
    boxes = torch.stack([O.decode(loc[i], pri) for i in range(B)])
    probs = F.softmax(conf, dim=2)
    out = detect_from_scores(_head(pri), boxes, probs, min_score, 0.45, 200)
    torch.cuda.synchronize()
    _check_exact(out, _oracle_stage(boxes, probs, min_score, 0.45, 200), 200)


def test_detect_fewer_than_topk_is_class_major_unsorted():
    from objectdetection_ssd_b200.head import detect_from_scores
    pri = H.priors()
    loc, conf = H.detect_inputs(32, 3, pri.shape[0], bg_bias=9.0)
    boxes = torch.stack([O.decode(loc[i], pri) for i in range(3)])
    probs = F.softmax(conf, dim=2)
    ref = _oracle_stage(boxes, probs, 0.05, 0.45, 200)
    assert all(0 < r[0].shape[0] <= 200 for r in ref), [r[0].shape for r in ref]
    out = detect_from_scores(_head(pri), boxes, probs, 0.05, 0.45, 200)
    torch.cuda.synchronize()
    _check_exact(out, ref, 200)


def test_detect_no_candidates_and_ties():
    from objectdetection_ssd_b200.head import detect_from_scores
    pri = H.priors()
    P = pri.shape[0]
    boxes = pri.unsqueeze(0).repeat(2, 1, 1).contiguous()
    probs = torch.zeros(2, P, 21)
    probs[0, :, 20] = 1.0                        # image 0: nothing above threshold -> 0 detections (Losses.py:62-63)
    probs[1, :, 20] = 0.4
    probs[1, :, 3] = 0.3                         # image 1: every prior ties at 0.3 in classes 3 and 7 (T5, T7)
    probs[1, :, 7] = 0.3
    out = detect_from_scores(_head(pri), boxes, probs, 0.2, 0.45, 200)
    torch.cuda.synchronize()
    ref = _oracle_stage(boxes, probs, 0.2, 0.45, 200)
    assert int(out["cnt"][0]) == 0 and ref[0][0].shape[0] == 0
    _check_exact(out, ref, 200)


def test_detect_small_topk_and_pixel_scale():
    from objectdetection_ssd_b200.head import detect_from_scores
    pri = H.priors()
    loc, conf = H.detect_inputs(33, 2, pri.shape[0], bg_bias=6.0)
    boxes = torch.stack([O.decode(loc[i], pri) for i in range(2)])
    probs = F.softmax(conf, dim=2)
    wh = torch.tensor([[500., 375.], [320., 480.]])
    out = detect_from_scores(_head(pri), boxes, probs, 0.01, 0.45, 17, img_wh=wh)
    torch.cuda.synchronize()
    ref = _oracle_stage(boxes, probs, 0.01, 0.45, 17)
    ref = [(rb * torch.tensor([w, h, w, h]), rc, rp, ri) for (rb, rc, rp, ri), (w, h) in zip(ref, wh.tolist())]
    _check_exact(out, ref, 17)


def test_detect_candidate_cap_overflow_is_flagged():
    from objectdetection_ssd_b200.head import detect_from_scores
    pri = H.priors()
    loc, conf = H.detect_inputs(34, 2, pri.shape[0], bg_bias=6.0)
    boxes = torch.stack([O.decode(loc[i], pri) for i in range(2)])
    probs = F.softmax(conf, dim=2)
    out = detect_from_scores(_head(pri), boxes, probs, 0.01, 0.45, 200, max_candidates=64)
    torch.cuda.synchronize()
    assert (out["cnt"].cpu() == -1).all()


def test_detect_ssd512_priors():
    from objectdetection_ssd_b200.head import detect_from_scores
    pri = H.priors("ssd512")
    loc, conf = H.detect_inputs(35, 1, pri.shape[0], bg_bias=7.0)
    boxes = torch.stack([O.decode(loc[0], pri)])
    probs = F.softmax(conf, dim=2)
    out = detect_from_scores(_head(pri), boxes, probs, 0.01, 0.45, 200)
    torch.cuda.synchronize()
    _check_exact(out, _oracle_stage(boxes, probs, 0.01, 0.45, 200), 200)


def test_detect_end_to_end_close():
    """The fused path (own decode + softmax): every emitted probability and box within its per-candidate bound of the
    float64 softmax / decode; detections equal the oracle's except where a boundary proof exists
    (tests/helpers.explain_detect_mismatches: probability within its error bound of min_score, a same-class IoU within
    IOU_REL of the threshold, or a bound-level order flip at the top-k cut).  Every difference must be explained; the
    number of differences is reported."""
    from objectdetection_ssd_b200.head import detect
    pri = H.priors()
    total = 0
    for seed, B, bias, min_score in ((36, 4, 7.0, 0.01), (37, 3, 6.0, 0.01), (38, 3, 8.0, 0.2)):
        loc, conf = H.detect_inputs(seed, B, pri.shape[0], bg_bias=bias)
        out = detect(_head(pri), loc, conf, min_score, 0.45, 200)
        torch.cuda.synchronize()
        total += H.compare_detect_with_oracle(out, loc, conf, pri, min_score, 0.45, 200, range(B))
    print(f"fused detect vs oracle: {total} detections differ, all with a boundary proof")


def _clustered_inputs(seed, B, pri, classes, jitter=0.02, frac=0.5):
    """Boxes = the priors with a small jitter (neighbouring priors overlap heavily -> strong suppression);
    probabilities only in ``classes`` for a random ``frac`` of the priors."""
    g = torch.Generator().manual_seed(seed)
    P = pri.shape[0]
    boxes = pri.unsqueeze(0).repeat(B, 1, 1).clone()
    boxes[..., :2] += jitter * torch.randn(B, P, 2, generator=g)
    boxes[..., 2:] *= torch.exp(jitter * torch.randn(B, P, 2, generator=g))
    probs = torch.zeros(B, P, 21)
    for c in classes:
        on = torch.rand(B, P, generator=g) < frac
        probs[..., c] = torch.where(on, 0.05 + 0.9 * torch.rand(B, P, generator=g), torch.zeros(()))
    probs[..., 20] = 1.0 - probs[..., :20].sum(-1).clamp(max=1.0)
    return boxes.contiguous(), probs.contiguous()


def test_detect_heavy_suppression_runs_through_every_slice():
    """Two classes, ~4.4k overlapping candidates each: the sweep needs many slices (the later ones larger than the
    shared-memory slice buffer -> global-memory path) and ends with fewer than top_k boxes (class-major output)."""
    from objectdetection_ssd_b200.head import detect_from_scores
    pri = H.priors()
    boxes, probs = _clustered_inputs(41, 2, pri, classes=(2, 11))
    ref = _oracle_stage(boxes, probs, 0.05, 0.45, 200)
    out = detect_from_scores(_head(pri), boxes, probs, 0.05, 0.45, 200)
    torch.cuda.synchronize()
    _check_exact(out, ref, 200)
    # the same candidates with a top_k small enough to stop early, and one large enough to need the whole list
    for tk in (1, 37, 600):
        out = detect_from_scores(_head(pri), boxes, probs, 0.05, 0.45, tk)
        torch.cuda.synchronize()
        _check_exact(out, _oracle_stage(boxes, probs, 0.05, 0.45, tk), tk)


def test_detect_quantised_scores_tie_across_classes_and_priors():
    """Probabilities rounded to multiples of 1/32: thousands of exact ties inside and across classes (T5, T7) and
    crowded sort bins."""
    from objectdetection_ssd_b200.head import detect_from_scores
    pri = H.priors()
    loc, conf = H.detect_inputs(42, 2, pri.shape[0], bg_bias=3.0)
    boxes = torch.stack([O.decode(loc[i], pri) for i in range(2)])
    probs = torch.round(F.softmax(conf, dim=2) * 32) / 32
    out = detect_from_scores(_head(pri), boxes, probs, 1 / 32, 0.45, 200)
    torch.cuda.synchronize()
    _check_exact(out, _oracle_stage(boxes, probs, 1 / 32, 0.45, 200), 200)


def test_detect_unaligned_prior_count_takes_the_plain_load_path():
    """P = 1001: image rows are not 16-byte aligned, so the score kernel cannot use its bulk copy."""
    from objectdetection_ssd_b200.head import detect_from_scores, detect
    pri = H.priors()[:1001].contiguous()
    loc, conf = H.detect_inputs(43, 3, 1001, bg_bias=3.0)
    boxes = torch.stack([O.decode(loc[i], pri) for i in range(3)])
    probs = F.softmax(conf, dim=2)
    out = detect_from_scores(_head(pri), boxes, probs, 0.02, 0.45, 50)
    torch.cuda.synchronize()
    _check_exact(out, _oracle_stage(boxes, probs, 0.02, 0.45, 50), 50)
    out2 = detect(_head(pri), loc, conf, 0.02, 0.45, 50)             # own softmax + decode on the same odd shape
    torch.cuda.synchronize()
    assert (out2["cnt"].cpu() == out["cnt"].cpu()).all()


def test_detect_randomised_differential():
    """Seeded random shapes, thresholds, top_k, tie densities and overlap densities (P not a multiple of 4 included):
    detections must equal the oracle's exactly (stage-isolated, so no expf boundary effects)."""
    from objectdetection_ssd_b200.head import MultiboxHead, detect_from_scores
    g = torch.Generator().manual_seed(2024)
    for trial in range(24):
        P = int(torch.randint(33, 2600, (1,), generator=g))
        B = int(torch.randint(1, 4, (1,), generator=g))
        top_k = [1, 5, 50, 200, 500][trial % 5]
        min_score = [0.01, 0.05, 0.3][trial % 3]
        iou_thr = [0.3, 0.45, 0.7][(trial // 3) % 3]
        ncls = [1, 3, 20][(trial // 2) % 3]                       # how many foreground classes are populated
        spread = [0.05, 0.3][(trial // 4) % 2]                   # small spread -> heavy overlap
        cx = 0.5 + spread * torch.randn(B, P, 2, generator=g)
        wh = 0.05 + 0.25 * torch.rand(B, P, 2, generator=g)
        boxes = torch.cat([cx, wh], 2).contiguous()
        probs = torch.zeros(B, P, 21)
        cls_ids = torch.randperm(20, generator=g)[:ncls]
        raw = torch.rand(B, P, ncls, generator=g) ** 3           # skewed towards small scores
        if trial % 4 == 1:
            raw = torch.round(raw * 16) / 16                     # exact ties
        probs[:, :, cls_ids] = raw * 0.9
        probs[..., 20] = 1.0 - probs[..., :20].max(-1).values
        pri = torch.cat([torch.rand(P, 2, generator=g), 0.1 + 0.2 * torch.rand(P, 2, generator=g)], 1)   # unused by from_scores
        out = detect_from_scores(MultiboxHead(pri, "cuda"), boxes, probs, min_score, iou_thr, top_k)
        torch.cuda.synchronize()
        ref = _oracle_stage(boxes, probs, min_score, iou_thr, top_k)
        try:
            _check_exact(out, ref, top_k)
        except AssertionError as e:
            raise AssertionError(f"trial {trial}: P={P} B={B} top_k={top_k} min_score={min_score} iou={iou_thr} ncls={ncls}: {e}")


def test_detect_suppression_chains_and_sparse_overlaps():
    """Hand-made chains inside one class and one slice: A suppresses B, B overlaps C but A does not -> C is KEPT
    (a suppressed box suppresses nobody, Losses.py:44-55); a candidate overlapping two higher-scored boxes of which
    only one survives; three mutually overlapping boxes (more recorded overlaps than the sparse sweep stores -> the
    general sweep); the same geometry in another class must not interact.  Exact against the oracle."""
    from objectdetection_ssd_b200.head import MultiboxHead, detect_from_scores
    P = 64
    g = torch.Generator().manual_seed(7)
    boxes = torch.zeros(1, P, 4)
    probs = torch.zeros(1, P, 21)
    probs[..., 20] = 1.0

    def put(i, cx, cy, w, h, cls, p):
        boxes[0, i] = torch.tensor([cx, cy, w, h])
        probs[0, i, cls] = p

    # chain along x: each box overlaps its neighbour (IoU 0.6) but not the one after (IoU 0.33 < 0.45)
    for k in range(6):
        put(k, 0.20 + 0.05 * k, 0.2, 0.2, 0.2, 3, 0.9 - 0.05 * k)          # kept: 0, 2, 4  (1 suppressed by 0, 3 by 2, ...)
    # the same chain in class 7, scores reversed
    for k in range(6):
        put(8 + k, 0.20 + 0.05 * k, 0.2, 0.2, 0.2, 7, 0.5 + 0.05 * k)
    # a box overlapping two higher-scored boxes, one of which is itself suppressed
    put(20, 0.60, 0.6, 0.2, 0.2, 5, 0.95)
    put(21, 0.65, 0.6, 0.2, 0.2, 5, 0.90)       # suppressed by 20
    put(22, 0.70, 0.6, 0.2, 0.2, 5, 0.85)       # overlaps 21 (suppressed) only -> kept
    put(23, 0.74, 0.6, 0.2, 0.2, 5, 0.80)       # overlaps 21 (0.38: no), 22 (0.67) -> suppressed by 22
    # four nearly identical boxes: every later one records three overlaps
    for k in range(4):
        put(30 + k, 0.3 + 0.002 * k, 0.7, 0.15, 0.15, 11, 0.7 - 0.01 * k)
    # background clutter in other classes, random small boxes
    for k in range(40, 64):
        put(k, float(torch.rand(1, generator=g)), float(torch.rand(1, generator=g)), 0.05, 0.05, int(torch.randint(12, 20, (1,), generator=g)), 0.3)
    pri = torch.cat([torch.rand(P, 2, generator=g), 0.1 + 0.2 * torch.rand(P, 2, generator=g)], 1)
    head = MultiboxHead(pri, "cuda")
    for top_k in (200, 5):
        out = detect_from_scores(head, boxes, probs, 0.05, 0.45, top_k)
        torch.cuda.synchronize()
        ref = _oracle_stage(boxes, probs, 0.05, 0.45, top_k)
        _check_exact(out, ref, top_k)
    kept3 = sorted(int(i) for i, c in zip(ref[0][3], ref[0][1]) if int(c) == 3) if top_k == 200 else None
    out = detect_from_scores(head, boxes, probs, 0.05, 0.45, 200)
    ids = out["prior"][0, :int(out["cnt"][0])].cpu().tolist()
    assert {0, 2, 4} <= set(ids) and not ({1, 3, 5} & set(ids)), ids
    assert {20, 22} <= set(ids) and not ({21, 23} & set(ids)), ids
