"""Detect on the outputs of a trained head, against the oracle and a float64 bound, on both detect routes.

The other detect tests draw conf from N(0, 1) plus a background bias and loc from 0.5 N(0, 1): thousands of mid-range
scores per image, almost no probability at 1.0, scattered boxes.  A trained head gives something else:

* saturated scores: a row whose other logits sit ~20 or more below its max has a probability of exactly 1.0f (in the
  kernels and in ATen), so an object brings hundreds to thousands of candidates that tie at 1.0, ordered only by
  (class, prior).  They all fall into coarse rank bin 0; more than SL = 2048 of them send the first slice through the
  global-memory block sweep, and the short list's sampled floor can land on bin 0 (floor = 1.0);
* collapsed boxes: the positive priors of an object regress to the same box, suppression is heavy and the output is
  often the class-major partition (fewer than top_k kept);
* images with few candidates, which never raise the floor.

Checks: stage-isolated (the oracle's fp32 boxes and probabilities in) bit for bit against ``O.detect_from_scores`` on
both routes; the fused path bit for bit on a family where its arithmetic provably equals ATen's, and within
per-candidate float64 bounds on ordinary trained margins; the short-list route's fallback count against a numpy
emulation of its score floor; threshold, score and IoU edges.
"""
import functools
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ssd_oracle as O
from objectdetection_ssd_b200 import synth
from tests import helpers as H
from tests.test_gpu_detect import _check_exact
from tests.test_gpu_detect_shortlist import _route
from tests.test_gpu_trained_regime import trained_conf

C = 21
NF = C - 1
BG = C - 1
LEVEL_COUNTS = (5776, 2166, 600, 150, 36, 4)
SL = 2048                        # slice keys sorted in shared memory (csrc/detect.cu)
SAMPLE_STRIDE = 35               # the short list's floor: every 35th row is sampled ...
SAMPLE_TARGET = 46               # ... and the floor is the highest coarse bin edge with 46 sampled candidates above it
CBINS = 256
KINDS = ("m10", "m17", "m25", "m40", "large", "multi", "few", "few")


# ----------------------------------------------------------------------------------------------------------- inputs
def _trained_image(seed, kind, pri):
    """One image of a trained head: gts, the oracle's class map, logits (trained_conf) and regressed offsets.

    m10 .. m40: synth.make_gt gts, background / class margins 10 .. 40, 1 % hard negatives, 10 % misclassified
    positives.  large: one object over most of the image; multi: four objects of three classes.  Both also light up
    every prior whose centre lies inside an object (a trained head fires there even where the prior's box matches the
    object poorly), margin 40 +- 25 %: thousands of probabilities of exactly 1.0.  few: one small object, no hard
    negatives: a few dozen candidates.  Positives regress to their gt (encode + 0.05 N(0, 1)), negatives N(0, 0.5)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    P = pri.shape[0]
    if kind == "large":
        gb = np.array([[0.06, 0.08, 0.94, 0.9]], np.float32)
        gc = np.array([7.0], np.float32)
    elif kind == "multi":
        gb = np.array([[0.04, 0.06, 0.46, 0.44], [0.55, 0.05, 0.95, 0.47], [0.06, 0.55, 0.45, 0.96],
                       [0.56, 0.54, 0.94, 0.92]], np.float32)
        gc = np.array([3.0, 11.0, 14.0, 3.0], np.float32)
    else:
        few = kind == "few"
        b, c = synth.make_gt(seed, 1, 1 if few else 2, 1 if few else 10)
        gb, gc = b[0], c[0]
        if few:                                   # a small object: few positives
            ctr = (gb[:, :2] + gb[:, 2:]) / 2
            gb = np.concatenate([ctr - 0.04, ctr + 0.04], 1).clip(0, 1).astype(np.float32)
    tb, tc = [torch.from_numpy(gb)], [torch.from_numpy(gc)]
    m = O.match_batch(tb, tc, O.cxcywh_to_xyxy(pri))
    cls = m["cls"][0].numpy().copy()
    obj = m["obj"][0].numpy().copy()
    if kind in ("large", "multi"):
        cx, cy = pri[:, 0].numpy(), pri[:, 1].numpy()
        for g, (box, c) in enumerate(zip(gb, gc)):
            sel = (cx > box[0]) & (cx < box[2]) & (cy > box[1]) & (cy < box[3]) & (cls == BG)
            cls[sel], obj[sel] = int(c), g
        conf = trained_conf(seed, cls[None], 40.0, spread=0.25, hard=0.01, mis=0.0)[0]
    elif kind == "few":
        conf = trained_conf(seed, cls[None], 25.0, hard=0.0, mis=0.1)[0]
    else:
        conf = trained_conf(seed, cls[None], float(kind[1:]), hard=0.01, mis=0.1)[0]
    tgt = O.encode(O.xyxy_to_cxcywh(tb[0])[torch.from_numpy(obj)], pri)
    pos = torch.from_numpy(cls != BG)
    loc = torch.from_numpy(rng.normal(0.0, 0.5, (P, 4)).astype(np.float32))
    loc[pos] = tgt[pos] + torch.from_numpy(rng.normal(0.0, 0.05, (int(pos.sum()), 4)).astype(np.float32))
    return loc, conf, cls


@functools.lru_cache(None)
def trained_batch(seed=1000, kinds=KINDS):
    """(priors, loc [B,P,4], conf [B,P,C], class map [B,P]) of one image per kind."""
    pri = H.priors()
    imgs = [_trained_image(seed + i, k, pri) for i, k in enumerate(kinds)]
    return (pri, torch.stack([a for a, _, _ in imgs]), torch.stack([b for _, b, _ in imgs]),
            np.stack([c for _, _, c in imgs]))


@functools.lru_cache(None)
def stage_inputs(seed=1000, kinds=KINDS):
    """The oracle's fp32 decoded boxes and probabilities of trained_batch: the stage-isolated inputs."""
    pri, loc, conf, _ = trained_batch(seed, kinds)
    boxes = torch.stack([O.decode(loc[i], pri) for i in range(loc.shape[0])])
    return pri, boxes, F.softmax(conf, dim=2)


def one_hot_family(seed=1000, kinds=KINDS):
    """Inputs on which the fused kernels' arithmetic provably equals ATen's: each row keeps the argmax of its trained
    logits and every other logit lies 105 to 145 below it, so exp(x - max) is 0 in both (ex2.approx.ftz flushes
    2^-151 and below; ATen's exp gives 0 below -104) and every softmax is exactly one-hot; the wh offsets are 0, so
    exp(0 / 5) = 1 on both sides and the centre decode is the same three IEEE operations (-fmad=false)."""
    pri, loc, conf, cls = trained_batch(seed, kinds)
    rng = np.random.Generator(np.random.PCG64(seed + 77))
    x = conf.numpy()
    top = x.max(-1, keepdims=True)
    oh = (top - rng.uniform(105.0, 145.0, x.shape)).astype(np.float32)
    arg = x.argmax(-1)
    np.put_along_axis(oh, arg[..., None], top, -1)
    loc = loc.clone()
    loc[..., 2:] = 0.0
    return pri, loc, torch.from_numpy(oh)


# ----------------------------------------------------------------------------------------------------------- oracle
@functools.lru_cache(None)
def _kept_all(key, min_score, iou_thr):
    boxes, probs = _CASES[key]()
    return [O.detect_from_scores(boxes[i], probs[i], min_score, iou_thr, 1 << 30) for i in range(boxes.shape[0])]


def oracle_topk(full, top_k):
    """O.detect_from_scores' output for ``top_k`` from its output for an unlimited top_k (the class-major list of every
    kept box): the same stable sort and cut as ssd_oracle.py:333-336.  The NMS, which does not depend on top_k, runs
    once per input."""
    b, c, p, i = full
    if b.shape[0] > top_k:
        p, order = torch.sort(p, dim=0, descending=True, stable=True)
        p, order = p[:top_k], order[:top_k]
        b, c, i = b[order], c[order], i[order]
    return b, c, p, i


def _stage_case():
    _, boxes, probs = stage_inputs()
    return boxes, probs


def _one_hot_case():
    pri, loc, conf = one_hot_family()
    return torch.stack([O.decode(loc[i], pri) for i in range(loc.shape[0])]), F.softmax(conf, dim=2)


def _one_hot_pair_case():
    boxes, probs = _one_hot_case()
    return boxes[PAIR], probs[PAIR]


PAIR = [4, 0]                    # the images of the min_score = 0 runs: the large object and a margin-10 image
_CASES = dict(stage=_stage_case, one_hot=_one_hot_case, one_hot_pair=_one_hot_pair_case)


def oracle(key, min_score, iou_thr, top_k):
    return [oracle_topk(f, top_k) for f in _kept_all(key, min_score, iou_thr)]


# ----------------------------------------------------------------------------------------------------------- short list
def coarse_rank(p):
    """csrc/detect.cu coarse_rank of fp32 probabilities >= 0: bin 0 = [1, ..), 32 bins per octave, 255 = the rest."""
    bits = np.asarray(p, np.float32).view(np.uint32).astype(np.int64)
    return np.clip((0x3F800000 >> 18) - (bits >> 18), 0, CBINS - 1)


def score_floor(probs_i, min_score):
    """The short list's score floor of one image (sample_floor, csrc/detect.cu), from its fp32 probabilities [P,C]:
    every SAMPLE_STRIDE-th row, the foreground probabilities >= min_score counted into the coarse bins, the first bin
    (from the top) at which SAMPLE_TARGET are reached; its lower edge is the floor if that is above min_score.
    Returns (floor, that bin or CBINS)."""
    ms = np.float32(min_score)
    rows = np.asarray(probs_i, np.float32)[::SAMPLE_STRIDE, :NF]
    h = np.bincount(coarse_rank(rows[rows >= ms]), minlength=CBINS)
    reach = np.nonzero(np.cumsum(h) >= SAMPLE_TARGET)[0]
    r = int(reach[0]) if reach.size else CBINS
    floor = ms
    if r < CBINS - 1:
        edge = np.uint32(((0x3F800000 >> 18) - r) << 18).view(np.float32)
        if edge > ms:
            floor = edge
    return floor, r


def route_kinds(probs, full, min_score, top_k):
    """Per image, how the short-list route serves it: 'not raised' (floor = min_score), 'decided' (the floor rose and
    per-class NMS on the candidates >= floor keeps more than top_k boxes) or 'fallback' (it keeps at most top_k: the
    sweep CTA lists the image again).  The kept boxes >= floor are the full NMS's kept boxes >= floor (a candidate's
    fate depends only on higher-scored ones).  Also returns each image's floor bin."""
    kinds, bins = [], []
    for i, (_, _, p, _) in enumerate(full):
        floor, r = score_floor(probs[i].numpy(), min_score)
        bins.append(r)
        if not floor > np.float32(min_score):
            kinds.append("not raised")
        else:
            kinds.append("decided" if int((p.numpy() >= floor).sum()) > top_k else "fallback")
    return kinds, bins


# ----------------------------------------------------------------------------------------------------------- GPU helpers
def _head(pri):
    from objectdetection_ssd_b200.head import MultiboxHead
    return MultiboxHead(pri, "cuda")


MAX_TOP_K = 1729                 # the largest top_k the sweep's shared memory holds with SSD300 (csrc/detect.cu)


def _big_top_k(full):
    """A top_k larger than the survivors of every image (the class-major partition), or the largest top_k the kernel
    takes when an image has more survivors than that."""
    return min(MAX_TOP_K, max(int(f[0].shape[0]) for f in full) + 1)


def _stage_run(head, boxes, probs, min_score, iou_thr, top_k, shortlist):
    from objectdetection_ssd_b200.head import detect_fallbacks, detect_from_scores
    with _route(shortlist):
        out = detect_from_scores(head, boxes, probs, min_score, iou_thr, top_k)
        nfb = detect_fallbacks(head, boxes.shape[0])
    return out, nfb


# ----------------------------------------------------------------------------------------------------------- CPU tests
def test_generator_saturates_and_collapses():
    """What the GPU tests rely on: the large object gives more than SL candidates at exactly 1.0 in one class (coarse
    bin 0), the multi image several classes tied at 1.0, the few images fewer candidates than can raise the floor;
    positives' decoded boxes collapse onto their object."""
    pri, boxes, probs = stage_inputs()
    fg = probs[..., :NF].numpy()
    ones = (fg == 1.0).sum(1)                                          # [B, NF]
    assert ones[4].max() > SL and int(ones[4].argmax()) == 7, ones[4]
    assert (ones[5] >= 100).sum() >= 3, ones[5]
    assert ((coarse_rank(fg[4]) == 0).sum()) > SL
    for i in (6, 7):
        assert int((fg[i] >= 0.01).sum()) < SAMPLE_STRIDE * SAMPLE_TARGET, i
    assert all(int((fg[i] == 1.0).sum()) > 0 for i in range(8) if KINDS[i] != "m10")
    # margins 10 .. 40: hard negatives and misclassified positives exist; more candidates at lower margins
    cand = (fg >= 0.01).sum((1, 2))
    assert cand[0] > cand[3] > 0, cand
    # collapsed boxes: the large object's kept list in class 7 is tiny
    full = _kept_all("stage", 0.01, 0.45)
    assert int((full[4][1] == 7).sum()) < 20


def test_one_hot_family_is_exact_in_aten():
    """ATen's fp32 softmax of the one-hot family is exactly 0 / 1 and its decode of zero wh offsets is the prior's
    size: the premise of the fused exact-equality tests."""
    pri, loc, conf = one_hot_family()
    p = F.softmax(conf, dim=2)
    assert bool(((p == 0) | (p == 1)).all()) and bool((p.sum(-1) == 1).all())
    gaps = conf.max(-1, keepdim=True).values - conf
    assert float(gaps[gaps > 0].min()) >= 104.0
    for i in range(loc.shape[0]):
        assert torch.equal(O.decode(loc[i], pri)[:, 2:], pri[:, 2:])
    assert int((p[..., :NF] == 1).sum()) > 5000


def test_float64_bounds_hold_for_aten_and_are_tight():
    """ATen's fp32 softmax and decode lie within the per-candidate bounds of helpers.softmax_f64 / decode_f64 on
    trained and N(0, 1) logits; the bounds stay within a few tens of ulp where the probability matters."""
    pri, loc, conf, _ = trained_batch()
    l2, c2 = H.detect_inputs(36, 2, pri.shape[0], bg_bias=7.0)
    for L, Cf in ((loc, conf), (l2, c2)):
        for i in range(L.shape[0]):
            p64, pb = H.softmax_f64(Cf[i].numpy())
            pa = F.softmax(Cf[i], dim=1).double().numpy()
            assert (np.abs(pa - p64) <= pb).all()
            b64, bb = H.decode_f64(L[i].numpy(), pri.numpy())
            ba = O.cxcywh_to_xyxy(O.decode(L[i], pri)).double().numpy()
            assert (np.abs(ba - b64) <= bb).all()
            big = p64 >= 1e-3
            d = np.abs(Cf[i].double().numpy() - Cf[i].double().numpy().max(-1, keepdims=True))
            assert (pb[big] <= p64[big] * H.EPS * (20 + 2 * d[big])).all()


def test_floor_emulation_sees_every_route_kind():
    """Over the stage-isolated runs (min_score 0.01 / 0.5 / 1.0, top_k 1 / 200 / all), the short list meets every kind
    of image: floor on bin 0, raised and decided, raised and not decided (fallback), and not raised."""
    _, _, probs = stage_inputs()
    seen, bin0 = set(), 0
    for ms in (0.01, 0.5, 1.0):
        full = _kept_all("stage", ms, 0.45)
        for tk in (1, 200, _big_top_k(full)):
            kinds, bins = route_kinds(probs, full, ms, tk)
            seen |= set(kinds)
            bin0 += sum(1 for k, r in zip(kinds, bins) if r == 0 and k != "not raised")
    assert seen == {"not raised", "decided", "fallback"}, seen
    assert bin0 > 0
    # min_score 0.01: the large object's and the multi image's floors are 1.0.  The large object keeps one box at 1.0
    # (its boxes collapse): not decided even at top_k = 1; the multi image is decided at top_k = 1, not at 200
    full = _kept_all("stage", 0.01, 0.45)
    k1, b1 = route_kinds(probs, full, 0.01, 1)
    k2, _ = route_kinds(probs, full, 0.01, 200)
    assert b1[4] == b1[5] == 0 and k1[4] == "fallback" and k1[5] == "decided" and k2[5] == "fallback", (b1, k1, k2)
    assert k1[6] == k1[7] == "not raised"


def test_big_top_k_exceeds_the_survivors():
    """The third top_k of the stage-isolated runs leaves every image but the margin-10 one at min_score 0.01 (4 447
    survivors) with fewer survivors than top_k: their output is the class-major partition."""
    for ms in (0.01, 0.5, 1.0):
        full = _kept_all("stage", ms, 0.45)
        n = [int(f[0].shape[0]) for f in full]
        tk = _big_top_k(full)
        assert all(k < tk for i, k in enumerate(n) if not (ms == 0.01 and i == 0)), (ms, n, tk)


def test_dyadic_pairs_have_iou_exactly_at_the_threshold():
    for thr in (0.5, 0.75):
        boxes, _, pair = _dyadic_pair_inputs(64, thr, 0)
        iou = O.iou_matrix(O.cxcywh_to_xyxy(boxes[0, pair[:1]]), O.cxcywh_to_xyxy(boxes[0, pair[1:]]))
        assert float(iou) == thr


# ----------------------------------------------------------------------------------------------------------- 2 + 5: stage-isolated
@pytest.mark.gpu
@pytest.mark.parametrize("min_score", [0.01, 0.5, 1.0])
def test_stage_isolated_trained_exact_on_both_routes(min_score):
    """The oracle's fp32 boxes / probabilities of the trained batch: both routes equal O.detect_from_scores bit for bit
    at top_k 1, 200 and above the survivors; the short-list route's fallback count equals the emulated one."""
    pri, boxes, probs = stage_inputs()
    head = _head(pri)
    full = _kept_all("stage", min_score, 0.45)
    for top_k in (1, 200, _big_top_k(full)):
        ref = oracle("stage", min_score, 0.45, top_k)
        kinds, _ = route_kinds(probs, full, min_score, top_k)
        for shortlist in (True, False):
            out, nfb = _stage_run(head, boxes, probs, min_score, 0.45, top_k, shortlist)
            _check_exact(out, ref, None, f"min_score {min_score} top_k {top_k} shortlist {shortlist}:")
            want = kinds.count("fallback") if shortlist else 0
            assert nfb == want, f"min_score {min_score} top_k {top_k}: {nfb} fallbacks, emulated {want} ({kinds})"


# ----------------------------------------------------------------------------------------------------------- 3: fused, exact
def _levels(t):
    out, s = [], 0
    for n in LEVEL_COUNTS:
        out.append(t[:, s:s + n].contiguous().cuda())
        s += n
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("min_score", [0.01, 0.0])
def test_fused_exact_family_every_entry_point(min_score):
    """One-hot logits and zero wh offsets: detect and detect_levels on both routes, SSDHeadContext.detect_host and a
    captured StaticHead.detect equal the oracle bit for bit; the short-list route's fallback count is the emulated one.
    min_score = 0 makes every (prior, class) a candidate, the zeros included (two images)."""
    from objectdetection_ssd_b200.ctx import SSDHeadContext, pinned_empty
    from objectdetection_ssd_b200.head import StaticHead, detect, detect_fallbacks, detect_levels
    pri, loc, conf = one_hot_family()
    key = "one_hot"
    if min_score == 0.0:
        loc, conf, key = loc[PAIR], conf[PAIR], "one_hot_pair"
    B, P = loc.shape[0], pri.shape[0]
    _, probs = _CASES[key]()
    head = _head(pri)
    full = _kept_all(key, min_score, 0.45)
    for top_k in (1, 200):
        ref = oracle(key, min_score, 0.45, top_k)
        kinds, _ = route_kinds(probs, full, min_score, top_k)
        for shortlist in (True, False):
            with _route(shortlist):
                a = detect(head, loc, conf, min_score, 0.45, top_k)
                na = detect_fallbacks(head, B)
                b = detect_levels(head, _levels(loc), _levels(conf), min_score, 0.45, top_k)
                nb = detect_fallbacks(head, B)
            what = f"min_score {min_score} top_k {top_k} shortlist {shortlist}"
            _check_exact(a, ref, None, what + " detect:")
            _check_exact(b, ref, None, what + " detect_levels:")
            want = kinds.count("fallback") if shortlist else 0
            assert na == want and nb == want, (what, na, nb, want, kinds)
    # the host context (top_k 200) and a captured StaticHead.detect on each route
    ref = oracle(key, min_score, 0.45, 200)
    ctx = SSDHeadContext(pri.numpy(), max_batch=B)
    hl, hc = pinned_empty(loc.shape), pinned_empty(conf.shape)
    hl[:] = loc.numpy()
    hc[:] = conf.numpy()
    ob, op = pinned_empty((B, 200, 4)), pinned_empty((B, 200))
    oc, oi, on = pinned_empty((B, 200), np.int32), pinned_empty((B, 200), np.int32), pinned_empty((B,), np.int32)
    ctx.detect_host(hl, hc, ob, op, oc, oi, on, min_score, 0.45)
    ctx.close()
    t = lambda a: torch.from_numpy(np.array(a))
    _check_exact(dict(boxes=t(ob), prob=t(op), cls=t(oc), prior=t(oi), cnt=t(on)), ref, None, "detect_host:")
    for shortlist in (True, False):
        sh = StaticHead(pri, B, B, "cuda")
        dl, dc = loc.cuda(), torch.full_like(conf, float("nan")).cuda()
        with _route(shortlist):
            sh.detect(dl, dc, min_score, 0.45, 200)                   # warm-up: allocates the workspace
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = sh.detect(dl, dc, min_score, 0.45, 200)
        dc.copy_(conf.cuda())
        g.replay()
        torch.cuda.synchronize()
        _check_exact(out, ref, None, f"captured StaticHead.detect shortlist {shortlist}:")
        del g


# ----------------------------------------------------------------------------------------------------------- 4: fused, bounds
@pytest.mark.gpu
@pytest.mark.parametrize("min_score", [0.01, 1e-6])
def test_fused_trained_margins_within_float64_bounds(min_score):
    """Ordinary trained logits: every probability and box the fused path emits lies within its per-candidate bound of
    the float64 softmax / decode, every difference from the oracle has a boundary proof, and both routes agree bit for
    bit.  At 1e-6 candidates lie up to ~14 below their row max, past the |x - max| <= 10 of a flat 16-ulp bound."""
    from objectdetection_ssd_b200.head import detect
    pri, loc, conf, _ = trained_batch()
    head = _head(pri)
    with _route(True):
        a = detect(head, loc, conf, min_score, 0.45, 200)
    with _route(False):
        b = detect(head, loc, conf, min_score, 0.45, 200)
    torch.cuda.synchronize()
    assert torch.equal(a["cnt"].cpu(), b["cnt"].cpu())
    for i, k in enumerate(a["cnt"].cpu().tolist()):
        for key in ("boxes", "prob", "cls", "prior"):
            assert torch.equal(a[key][i, :k].cpu(), b[key][i, :k].cpu()), f"image {i}: {key} differs between the routes"
    n = H.compare_detect_with_oracle(a, loc, conf, pri, min_score, 0.45, 200, range(loc.shape[0]))
    if min_score == 1e-6:
        d = conf.max(-1, keepdim=True).values - conf
        p = F.softmax(conf, dim=2)
        assert float(d[..., :NF][p[..., :NF] >= min_score].max()) > 10.0
    print(f"min_score {min_score}: {n} detections differ from the oracle, all with a boundary proof")


# ----------------------------------------------------------------------------------------------------------- 5: automatic route
@pytest.mark.gpu
def test_batch_128_automatic_route_equals_exhaustive_and_counts_fallbacks():
    """128 trained images (the automatic choice takes the short list from ~900 k rows): bit for bit the forced
    exhaustive route, and as many fallbacks as the emulation predicts (stage-isolated, where the probabilities are
    known exactly)."""
    from objectdetection_ssd_b200.head import detect, detect_fallbacks, detect_from_scores
    pri, loc, conf, _ = trained_batch(2000, KINDS * 16)
    _, boxes, probs = stage_inputs(2000, KINDS * 16)
    head = _head(pri)
    B = loc.shape[0]
    old = os.environ.pop("SSDHEAD_DETECT_SHORTLIST", None)
    try:
        auto = detect(head, loc, conf, 0.01, 0.45, 200)
        sauto = detect_from_scores(head, boxes, probs, 0.01, 0.45, 200)
        nfb = detect_fallbacks(head, B)
    finally:
        if old is not None:
            os.environ["SSDHEAD_DETECT_SHORTLIST"] = old
    with _route(False):
        full = detect(head, loc, conf, 0.01, 0.45, 200)
        sfull = detect_from_scores(head, boxes, probs, 0.01, 0.45, 200)
    torch.cuda.synchronize()
    for x, y in ((auto, full), (sauto, sfull)):
        assert torch.equal(x["cnt"].cpu(), y["cnt"].cpu())
        for i, k in enumerate(x["cnt"].cpu().tolist()):
            for key in ("boxes", "prob", "cls", "prior"):
                assert torch.equal(x[key][i, :k].cpu(), y[key][i, :k].cpu()), f"image {i}: {key}"
    kept = [O.detect_from_scores(boxes[i], probs[i], 0.01, 0.45, 1 << 30) for i in range(B)]
    kinds, _ = route_kinds(probs, kept, 0.01, 200)
    assert nfb == kinds.count("fallback") > 0, (nfb, kinds.count("fallback"))
    _check_exact(sauto, [oracle_topk(f, 200) for f in kept], None, "batch 128:")


# ----------------------------------------------------------------------------------------------------------- 6: edges
def _small_stage(P=1536, first=2000):
    """Two trained images (a margin-10 one and the multi one) cut to priors [first, first + P): cheap oracle runs at
    min_score <= 0, where every (prior, class) is a candidate."""
    _, boxes, probs = stage_inputs()
    sel = slice(first, first + P)
    return boxes[[0, 5], sel].contiguous(), probs[[0, 5], sel].contiguous()


def _run_both(head, boxes, probs, min_score, iou_thr, top_k, what):
    ref = [O.detect_from_scores(boxes[i], probs[i], min_score, iou_thr, top_k) for i in range(boxes.shape[0])]
    for shortlist in (True, False):
        out, _ = _stage_run(head, boxes, probs, min_score, iou_thr, top_k, shortlist)
        _check_exact(out, ref, None, f"{what} shortlist {shortlist}:")
    return ref


@pytest.mark.gpu
def test_min_score_edges():
    """min_score 0, a score present exactly, 1.0, nextafter(1, 2), -1 and NaN, against the oracle on both routes."""
    boxes, probs = _small_stage()
    head = _head(torch.rand(boxes.shape[1], 4))
    kept = O.detect_from_scores(boxes[0], probs[0], 0.01, 0.45, 1 << 30)[2]
    present = float(torch.sort(kept, descending=True).values[100])         # a kept box stays kept at a higher min_score
    for ms in (0.0, present, 1.0, float(np.nextafter(np.float32(1), np.float32(2))), -1.0, float("nan")):
        ref = _run_both(head, boxes, probs, ms, 0.45, 200, f"min_score {ms!r}")
        if ms == present:
            assert any(bool((r[2] == present).any()) for r in ref)
        if ms > 1.0 or ms != ms:
            assert all(r[0].shape[0] == 0 for r in ref)


@pytest.mark.gpu
@pytest.mark.parametrize("iou_thr", [0.0, 1.0, 1.5, -0.1, float("nan")])
def test_iou_threshold_edges(iou_thr):
    """iou_thr 0 (every same-class box with IoU >= 0 goes), 1, 1.5 and -0.1 and NaN, against the oracle on both routes,
    on the full trained batch (the large object's > 2048 ties included)."""
    pri, boxes, probs = stage_inputs()
    head = _head(pri)
    for top_k in (200, 1000):
        _run_both(head, boxes, probs, 0.01, iou_thr, top_k, f"iou_thr {iou_thr} top_k {top_k}")


def _dyadic_pair_inputs(P, thr, n_ties):
    """A pair of class-0 boxes whose IoU is exactly ``thr`` (dyadic corners: every fp32 operation is exact), scores 1.0
    at priors 0 and 1 - the first two keys of the sweep.  The lower one must be suppressed (IoU >= thr).  ``n_ties``
    more candidates at 1.0 in class 1 (all on one box) make coarse bin 0, and so the first slice, larger than SL: the
    pair is then swept by the global-memory block path (iou_ge) instead of the shared-memory sweep (iou_ge_fast).
    Every other prior is background."""
    boxes = torch.zeros(1, P, 4)
    boxes[0, :, :2] = 0.5
    boxes[0, :, 2:] = 0.125
    probs = torch.zeros(1, P, C)
    probs[0, :, BG] = 1.0
    # A = [0.25, 0.25] - [0.75, 0.75] (area 1/4); B shares its left, bottom and right edges and has height thr / 2
    # (area thr / 4, inside A): IoU = (thr / 4) / (1 / 4) = thr
    boxes[0, 0] = torch.tensor([0.5, 0.5, 0.5, 0.5])
    boxes[0, 1] = torch.tensor([0.5, 0.25 + thr / 4, 0.5, thr / 2])
    probs[0, :2, BG] = 0.0
    probs[0, :2, 0] = 1.0
    for j in range(2, 2 + n_ties):
        probs[0, j, BG] = 0.0
        probs[0, j, 1] = 1.0
    # a few other class-0 boxes just below 1.0, disjoint from the pair
    for j, x in zip(range(2 + n_ties, 6 + n_ties), (0.0625, 0.9375, 0.0625, 0.9375)):
        boxes[0, j] = torch.tensor([x, 0.0625 if j % 2 else 0.9375, 0.0625, 0.0625])
        probs[0, j, BG] = 0.0
        probs[0, j, 0] = 0.5
    return boxes.contiguous(), probs.contiguous(), [0, 1]


@pytest.mark.gpu
@pytest.mark.parametrize("thr", [0.5, 0.75])
@pytest.mark.parametrize("n_ties", [0, 2100])
def test_iou_exactly_at_threshold(thr, n_ties):
    """IoU == iou_thr suppresses (the reference's `>=`), in the shared-memory sweep (n_ties = 0) and in a first slice
    larger than SL (n_ties = 2100), on both routes."""
    P = 64 if n_ties == 0 else 2304
    boxes, probs, pair = _dyadic_pair_inputs(P, thr, n_ties)
    head = _head(torch.rand(P, 4))
    ref = _run_both(head, boxes, probs, 0.01, thr, 200, f"thr {thr} ties {n_ties}")
    kept = set(ref[0][3].tolist())
    assert 0 in kept and 1 not in kept, kept


@pytest.mark.gpu
def test_signed_zero_negative_and_large_scores():
    """detect_from_scores with -0.0 (ties with +0.0), negative scores (rank below zero) and scores above 1 (rank above
    1.0), at min_score 0, -1 and -inf, against the oracle on both routes.  A -0.0 score must not come first."""
    boxes, probs = _small_stage(P=1024)
    probs = probs.clone()
    g = torch.Generator().manual_seed(5)
    B, P = probs.shape[:2]
    for b in range(B):
        rows = torch.randperm(P, generator=g)[:300]
        cls = torch.randint(0, NF, (300,), generator=g)
        vals = torch.cat([torch.full((100,), -0.0), -torch.rand(100, generator=g),
                          1.0 + 3 * torch.rand(90, generator=g), torch.tensor([float("inf")] * 5 + [-float("inf")] * 5)])
        probs[b, rows, cls] = vals
    head = _head(torch.rand(P, 4))
    for ms in (0.0, -1.0, -float("inf")):
        for top_k in (1, 200, 1500):
            ref = _run_both(head, boxes, probs, ms, 0.45, top_k, f"min_score {ms} top_k {top_k}")
    # top_k = 1 at min_score 0: the detection is a score > 1, never -0.0
    out, _ = _stage_run(head, boxes, probs, 0.0, 0.45, 1, True)
    assert bool((out["prob"][:, 0] > 1.0).all())


@pytest.mark.gpu
def test_fused_nonfinite_logits_and_extreme_offsets():
    """The one-hot family with NaN, +inf and -inf logits, +-1e4 rows, wh offsets of +450 (exp overflows: infinite
    boxes), -450 (denormal widths), -530 (exp underflows to 0) and NaN offsets: both routes equal the oracle bit for bit
    (NaN boxes compare equal to NaN)."""
    from objectdetection_ssd_b200.head import detect
    pri, loc, conf = one_hot_family()
    loc, conf = loc[[4, 5]].clone(), conf[[4, 5]].clone()           # the large object and the multi image: thousands of foreground rows
    rng = np.random.Generator(np.random.PCG64(31))
    P = pri.shape[0]
    fgrows = [np.nonzero((conf[b, :, :NF].max(-1).values >= conf[b, :, BG]).numpy())[0] for b in range(2)]
    for b in range(2):
        r = rng.permutation(fgrows[b])
        conf[b, r[0:20], 5] = float("nan")
        conf[b, r[20:40], 2] = float("inf")
        conf[b, r[40:60], 9] = -float("inf")
        conf[b, r[60:80]] = torch.from_numpy(1e4 * rng.choice([-1.0, 1.0], (20, C)).astype(np.float32))
        loc[b, r[80:100], 2] = 450.0
        loc[b, r[100:120], 3] = -450.0
        loc[b, r[120:140], 2:] = -530.0
        loc[b, r[140:150], int(rng.integers(0, 4))] = float("nan")
    head = _head(pri)
    for top_k in (1, 200):
        ref = [O.detect_image(loc[b], conf[b], pri, 0.01, 0.45, top_k) for b in range(2)]
        if top_k == 200:
            assert any(bool(torch.isinf(r[0]).any()) for r in ref) and any(bool(torch.isnan(r[0]).any()) for r in ref)
        for shortlist in (True, False):
            with _route(shortlist):
                out = detect(head, loc, conf, 0.01, 0.45, top_k)
            _check_exact(out, ref, None, f"top_k {top_k} shortlist {shortlist}:")


def test_boundary_proof_covers_order_flips_at_one_and_nothing_else():
    """Margin-17 image 1: priors 6379 and 6487 of class 16 both get probability 1.0 in ATen (float64: 1 - 9e-8 and
    1 - 8e-9, inside each other's error bounds) and overlap (IoU 0.95).  ATen's tie keeps the lower prior; an fp32
    softmax that rounds 6379's probability to the float below 1.0 keeps 6487 instead.  The boundary proof accepts that
    swap; dropping a detection of a class with no such pair, or adding one, stays unexplained."""
    pri, loc, conf, _ = trained_batch()
    rb, rc, rp, ri = O.detect_image(loc[1], conf[1], pri, 0.01, 0.45, 200)
    ref = {(int(c), int(p)) for c, p in zip(rc, ri)}
    assert (16, 6379) in ref and (16, 6487) not in ref
    swapped = (ref - {(16, 6379)}) | {(16, 6487)}
    n, unexplained = H.explain_detect_mismatches(loc[1], conf[1], pri, 0.01, 0.45, 200, swapped, ref)
    assert n == 2 and not unexplained
    p = F.softmax(conf[1], dim=1)
    lone = [(c, q) for c, q in ref if c != 16 and 0.05 < float(p[q, c]) < 0.99]
    for c, q in lone[:5]:
        n, unexplained = H.explain_detect_mismatches(loc[1], conf[1], pri, 0.01, 0.45, 200, ref - {(c, q)}, ref)
        if unexplained:
            break
    else:
        raise AssertionError(f"every dropped detection was explained: {lone[:5]}")
