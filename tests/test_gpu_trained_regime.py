"""The training step on the logits of a trained head, against a float64 reference.

The other loss tests draw conf from N(0, 1): every per-row cross entropy (CE) lies between about 0.5 and 6 and ties are
rare.  A head a few epochs into training gives background margins of 10 to 40: most negative rows have a CE below 1e-5
or exactly 0 in fp32, and the positives' CE spans 1e-7 to 30.  There the mining ranks positives (value 0) together
with zero-CE negatives, a dropped mined row changes the conf loss by ~1e-7 relative, and a mined row's gradient is
~1e-10 / N.  So the checks here are exact or scaled to the values:

* mined set: the oracle's rule (``O.mine_hard_negatives``) applied to the kernel's own CE tap reproduces the kernel's
  ``mined_mask`` bit for bit; which selection path each image takes is computed from the taps and asserted;
* CE: within ``ce_bound`` of the float64 CE (derived below), which the ATen fp32 oracle must meet as well;
* sums: ``sums[1]`` is the float64 sum of the taps over positives and mined rows, ``sums[0]`` the float64 L1 within its
  rounding budget; ``losses`` are the fp32 quotients of the sums;
* gradients: row by row against the float64 closed form under a bound scaled by the row's softmax and 1/N;
* routes: the flat step, the per-level step, the context's resident step and the three-kernel route give the same bits.

A gt labelled ``C - 1`` is a background gt, as in the reference: the priors it wins are negatives.  Non-finite ``loc``
is out of scope: the kernel takes sign(NaN) = 0 for the loc gradient where autograd gives NaN.
"""
import numpy as np
import pytest
import torch

from objectdetection_ssd_b200 import synth
from oracle import ssd_oracle as O
from tests import helpers as H

C = 21
BG = C - 1
EPS = 2.0 ** -23                 # one ulp of fp32 relative to the value, at most
LEVEL_COUNTS = (5776, 2166, 600, 150, 36, 4)


# ----------------------------------------------------------------------------------------------------------- reference
def ce_f64(conf, cls):
    """float64 CE of every row of the fp32 logits ``conf`` [..., C] against ``cls`` [...] (int)."""
    x = np.asarray(conf, np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        m = x.max(-1, keepdims=True)
        d = x - m
        lse = np.log(np.exp(d).sum(-1))
        return lse - np.take_along_axis(d, np.asarray(cls)[..., None], -1)[..., 0]


def ce_bound(conf, ce64):
    """Bound on |CE_fp32 - CE_f64| for rows of fp32 logits, of the form abs + rel * CE.

    The streaming kernel computes s = sum_q exp(d_q), d_q = x_q - max, and CE = log(s) - d_c (csrc/loss.cu,
    row_cross_entropy).  Each exp goes through ex2.approx.ftz with a relative error <= (2 + 1.16|d|) ulp
    (loss.cu:66-67); the fp32 rounding of d_q itself adds |d_q| / 2 ulp, so term q is off by at most
    (2 + 2|d_q|) eps e^{d_q}, and terms below 2^-126 are flushed (absolute C 2^-126).  The C - 1 additions each
    round by half an ulp of a partial sum <= s.  Relative to s (>= 1, the max term is exactly 1):
        abs = eps (2 + 2 X + (C - 1) / 2 + |log s|) + C 2^-126,    X = sum_q |d_q| e^{d_q} / s,
    where |log s| eps covers logf.  The rounding of d_c and of the final subtraction add eps / 2 each of |d_c| <= CE:
        rel = eps.
    For a trained negative (X ~ 1e-4) that is ~1.5e-6 absolute; the ~2e-7 of loss.cu:66-67 is the exp part alone.
    ATen's fp32 log_softmax (1-ulp exp, another summation order) stays inside the same bound."""
    x = np.asarray(conf, np.float64)
    m = x.max(-1, keepdims=True)
    d = x - m
    e = np.exp(d)
    s = e.sum(-1)
    X = (np.abs(d) * e).sum(-1) / s
    ab = EPS * (2.0 + 2.0 * X + (C - 1) / 2.0 + np.abs(np.log(s))) + C * 2.0 ** -126
    return ab + EPS * np.abs(ce64)


def reference_f64(loc, conf, ref, mined):
    """float64 loss of the fp32 inputs on the oracle's (exact) match and the given mined set [B,P] bool.
    Returns dict(ce (assigned class), ce_bg, sums (l1, ce), N, grad_loc, grad_conf, grad_bound)."""
    x = conf.double().numpy()
    cls = ref["cls"].numpy()
    pos = ref["pos"].numpy()
    mined = np.asarray(mined)
    N = int(pos.sum())
    ce = ce_f64(x, cls)
    ce_bg = ce_f64(x, np.full(cls.shape, BG))
    tgt = ref["target"].double().numpy()                      # fp32 targets (oracle encode), positives in row order
    dl = loc.double().numpy()[pos] - tgt
    l1 = np.abs(dl).sum()
    sel = pos | mined
    with np.errstate(invalid="ignore", over="ignore"):
        sum_ce = ce[pos].sum() + ce[mined].sum()
        m = x.max(-1, keepdims=True)
        d = x - m
        e = np.exp(d)
        p = e / e.sum(-1, keepdims=True)
    onehot = np.zeros_like(p)
    np.put_along_axis(onehot, cls[..., None], 1.0, -1)
    gc = np.where(sel[..., None], (p - onehot) / N, 0.0)
    # fp32 softmax: expf (2 ulp), 20 additions, 1/s and the product: <= 16 eps relative, plus |d| eps from d's rounding;
    # then p - onehot, fl(1/N) and the product: eps / 2 each of the result.  Rows that carry no gradient must be exactly
    # zero.
    with np.errstate(invalid="ignore"):
        gb = np.where(sel[..., None], (EPS * ((16.0 + 2.0 * np.abs(d)) * p + 2.0 * np.abs(p - onehot))) / N + 1e-44, 0.0)
    gl = np.zeros(loc.shape, np.float64)
    gl[pos] = np.sign(dl) / (4.0 * N)
    return dict(ce=ce, ce_bg=ce_bg, sums=(l1, sum_ce), N=N, grad_loc=gl, grad_conf=gc, grad_bound=gb, dl=dl, tgt=tgt)


# ----------------------------------------------------------------------------------------------------------- inputs
def trained_conf(seed, cls, margin, spread=0.5, hard=0.01, mis=0.1, scale=1.0, huge_rows=0, bf16=False):
    """Logits of a trained head for the class map ``cls`` [B,P] (int): N(0,1) noise, the assigned class raised by
    margin * U(1 - spread, 1 + spread); a fraction ``hard`` of the negatives has a foreground class 0.1-4 above the
    background (hard negatives), a fraction ``mis`` of the positives the background 0.1-8 above their class
    (misclassified).  Then scaled by ``scale``; ``huge_rows`` rows per image set to +-1e4; optionally bf16-quantised."""
    rng = np.random.Generator(np.random.PCG64(seed))
    B, P = cls.shape
    conf = rng.standard_normal((B, P, C), dtype=np.float32)
    mrow = (margin * rng.uniform(1 - spread, 1 + spread, (B, P))).astype(np.float32)
    bi, pi = np.meshgrid(np.arange(B), np.arange(P), indexing="ij")
    conf[bi, pi, cls] += mrow
    neg = cls == BG
    hn = neg & (rng.random((B, P)) < hard)
    fg = rng.integers(0, BG, (B, P))
    conf[hn, fg[hn]] = conf[hn, BG] + rng.uniform(0.1, 4.0, int(hn.sum())).astype(np.float32)
    mp = ~neg & (rng.random((B, P)) < mis)
    conf[mp, BG] = conf[mp, cls[mp]] + rng.uniform(0.1, 8.0, int(mp.sum())).astype(np.float32)
    if scale != 1.0:
        conf *= np.float32(scale)
    for b in range(B):
        rows = rng.choice(P, huge_rows, replace=False)
        conf[b, rows] = np.float32(1e4) * rng.choice(np.array([-1.0, 1.0], np.float32), (huge_rows, C))
    t = torch.from_numpy(conf)
    return t.bfloat16().float() if bf16 else t


def class_map(pri, tb, tc, pos_iou=0.5):
    return O.match_batch(tb, tc, O.cxcywh_to_xyxy(pri), pos_iou)["cls"].numpy()


def case_inputs(name, seed=0, B=4):
    """The trained-head families: margins 10 / 17 / 25 / 40, logits at |x| ~ 200 with +-1e4 rows, bf16 logits."""
    pri = H.priors()
    P = pri.shape[0]
    gb, gc = synth.make_gt(700 + seed, B, 2, 10)
    tb = [torch.from_numpy(b) for b in gb]
    tc = [torch.from_numpy(c) for c in gc]
    loc = torch.from_numpy(synth.make_head(700 + seed, B, P)[0])
    cls = class_map(pri, tb, tc)
    kind, _, arg = name.partition("_")
    if kind == "margin":
        conf = trained_conf(seed, cls, float(arg))
    elif kind == "scaled":
        conf = trained_conf(seed, cls, 10.0, scale=20.0, huge_rows=3)
    elif kind == "bf16":
        conf = trained_conf(seed, cls, 17.0, bf16=True)
    else:
        raise ValueError(name)
    return pri, loc, conf, tb, tc


CASES = ["margin_10", "margin_17", "margin_25", "margin_40", "scaled", "bf16"]


def keys_of(ce_tap, pos):
    """The mining keys the kernel ranks: CE bits without the sign, 0 for positives (uint32 [B,P])."""
    k = np.asarray(ce_tap, np.float32).view(np.uint32) & np.uint32(0x7fffffff)
    return np.where(np.asarray(pos), np.uint32(0), k)


def selection_path(key, k):
    """Which selection the mining kernel takes for one image (csrc/loss.cu, mine_body step 2), emulated in numpy
    float32: ("all"|"none", ...), ("fast", boundary bin, its count), or ("radix", T) with T the k-th largest key."""
    P = key.shape[0]
    if k >= P:
        return ("all",)
    if k == 0:
        return ("none",)
    kmax = int(key.max())
    if 0 < kmax < 0x7f800000:
        vmax = np.uint32(kmax).view(np.float32)
        scale = np.float32(2047.0) / vmax
        bins = (key.view(np.float32) * scale).astype(np.float32).astype(np.int64)
        assert bins.max() <= 2047, "a key above the histogram range"
        hist = np.bincount(bins, minlength=2048)
        above = np.cumsum(hist[::-1])[::-1]                       # keys in bin >= i
        bq = int(np.nonzero(above >= k)[0].max())
        if hist[bq] <= 512:
            return ("fast", bq, int(hist[bq]))
    return ("radix", int(np.sort(key)[::-1][k - 1]))


def kernel_rank_positives_in(key, pos, mined, k):
    """True when positives (key 0) took ranks among the zero-key rows the image mined (ties to the lower index)."""
    z = np.nonzero(mined & (key == 0))[0]
    return z.size > 0 and bool((np.nonzero(pos)[0] < z.max()).any())


# ----------------------------------------------------------------------------------------------------------- routes
def _head(pri):
    from objectdetection_ssd_b200.head import MultiboxHead
    return MultiboxHead(pri, "cuda")


def three_kernel_route(head, loc, conf, gt, neg_ratio, pos_iou):
    """ssdhead_ce_match_stream + finaliser + ssdhead_mine: the keys are built after the forced match."""
    from objectdetection_ssd_b200 import _lib
    B, P = int(loc.shape[0]), head.P
    m = head._match_outputs(gt, False)
    ws = head._workspace(_lib.WS_LOSS, B, 0)
    wm = head._workspace(_lib.WS_MATCH, B, gt.sumG)
    st = torch.cuda.current_stream().cuda_stream
    gl, gcf = torch.empty_like(loc), torch.empty_like(conf)
    ce = torch.empty(B, P, device="cuda")
    mined = torch.empty(B, (P + 31) // 32, dtype=torch.int32, device="cuda")
    sums = torch.empty(2, dtype=torch.float64, device="cuda")
    losses = torch.empty(2, device="cuda")
    lib = head.lib
    _lib.check(lib.ssdhead_ce_match_stream(conf.data_ptr(), gt.boxes.data_ptr(), gt.classes.data_ptr(), gt.off.data_ptr(),
                                           head.pri_xyxy.data_ptr(), B, P, C, gt.sumG, float(pos_iou), ce.data_ptr(),
                                           gl.data_ptr(), gcf.data_ptr(), m["cls_u8"].data_ptr(), m["best_prior"].data_ptr(),
                                           m["npos"].data_ptr(), ws.data_ptr(), ws.numel(), wm.data_ptr(), wm.numel(), 1, st),
               "ssdhead_ce_match_stream")
    _lib.check(lib.ssdhead_mine(loc.data_ptr(), conf.data_ptr(), gt.boxes.data_ptr(), gt.classes.data_ptr(), gt.off.data_ptr(),
                                head.pri_xyxy.data_ptr(), head.pri_cxcywh.data_ptr(), m["best_prior"].data_ptr(),
                                m["npos"].data_ptr(), m["npos"][B:].data_ptr(), m["cls_u8"].data_ptr(), B, P, C,
                                int(neg_ratio), float(pos_iou), sums.data_ptr(), losses.data_ptr(), gl.data_ptr(),
                                gcf.data_ptr(), mined.data_ptr(), ce.data_ptr(), ws.data_ptr(), ws.numel(), st),
               "ssdhead_mine")
    return dict(losses=losses, sums=sums, grad_loc=gl, grad_conf=gcf, ce=ce, mined_mask=mined, npos=m["npos"],
                cls_u8=m["cls_u8"])


def run_routes(pri, loc, conf, tb, tc, neg_ratio=3, pos_iou=0.5, levels=True, resident=True):
    """Every single-GPU route of the training step on the same inputs.  Returns {route: outputs}."""
    from objectdetection_ssd_b200.ctx import SSDHeadContext
    from objectdetection_ssd_b200.head import PackedGT
    head = _head(pri)
    B, P = int(loc.shape[0]), pri.shape[0]
    l, c = loc.cuda().contiguous(), conf.cuda().contiguous()
    gt = PackedGT(tb, tc, head.dev)
    out = dict(flat=head.loss(l, c, gt, with_grads=True, taps=True, neg_ratio=neg_ratio, pos_iou=pos_iou))
    out["three"] = three_kernel_route(head, l, c, gt, neg_ratio, pos_iou)
    if levels:
        counts = LEVEL_COUNTS if P == sum(LEVEL_COUNTS) else (P // 2, P - P // 2)
        bounds = np.cumsum((0,) + tuple(counts))
        lv = head.loss_levels([l[:, a:b].contiguous() for a, b in zip(bounds[:-1], bounds[1:])],
                              [c[:, a:b].contiguous() for a, b in zip(bounds[:-1], bounds[1:])],
                              gt, with_grads=True, neg_ratio=neg_ratio, pos_iou=pos_iou)
        out["levels"] = dict(losses=lv["losses"], sums=lv["sums"], grad_loc=torch.cat(lv["grad_loc"], 1),
                             grad_conf=torch.cat(lv["grad_conf"], 1))
    if resident:
        ctx = SSDHeadContext(pri.numpy(), max_batch=B)
        st = torch.cuda.current_stream().cuda_stream
        gl = torch.full_like(l, 3.0)
        gcf = torch.full_like(c, -1.0)
        sums = torch.empty(2, dtype=torch.float64, device="cuda")
        losses = torch.empty(2, device="cuda")
        ctx.loss_dev_resident(l.data_ptr(), c.data_ptr(), gt.boxes.data_ptr(), gt.classes.data_ptr(), gt.off.data_ptr(),
                              B, gt.sumG, sums.data_ptr(), losses.data_ptr(), gl.data_ptr(), gcf.data_ptr(), st, fresh=True,
                              neg_ratio=neg_ratio, pos_iou=pos_iou)
        torch.cuda.synchronize()
        ctx.close()
        out["resident"] = dict(losses=losses, sums=sums, grad_loc=gl, grad_conf=gcf)
    torch.cuda.synchronize()
    return {name: {k: (v.cpu() if torch.is_tensor(v) else v) for k, v in o.items()} for name, o in out.items()}


def same_bits(a, b):
    if a.dtype == torch.float64:
        return torch.equal(a.view(torch.int64), b.view(torch.int64))
    return torch.equal(a.view(torch.int32), b.view(torch.int32))


def assert_routes_agree(outs):
    f = outs["flat"]
    for name, o in outs.items():
        for key in ("losses", "sums", "grad_loc", "grad_conf"):
            assert same_bits(o[key], f[key]), f"{name} route: {key} differs from the flat step"
    assert same_bits(outs["three"]["ce"], f["ce"]), "three-kernel route: CE taps differ from the flat step"
    for key in ("mined_mask", "cls_u8", "npos"):
        assert torch.equal(outs["three"][key], f[key]), f"three-kernel route: {key} differs from the flat step"


# ----------------------------------------------------------------------------------------------------------- checks
def check_against_references(pri, loc, conf, tb, tc, o, neg_ratio=3, pos_iou=0.5, finite_rows=None):
    """The tap-based checks of one route's outputs ``o`` (flat step or three-kernel route).  Returns a dict of
    per-image selection paths and the float64 reference."""
    ref = O.multibox_loss(loc, conf, tb, tc, pri, thr=pos_iou, ratio=neg_ratio)
    B, P = conf.shape[:2]
    pos = ref["pos"]
    assert torch.equal(o["cls_u8"].long(), ref["cls"]), "class map"
    assert torch.equal(o["npos"][:B].long(), ref["npos"]), "positives per image"
    ce_tap = o["ce"]
    mined = H.unpack_mask(o["mined_mask"], P)
    # the mined set, exactly: the oracle's rule on the kernel's own CE
    assert torch.equal(mined, O.mine_hard_negatives(ce_tap, pos, neg_ratio)), "mined set differs from the rule on the taps"
    key = keys_of(ce_tap.numpy(), pos.numpy())
    paths = []
    for b in range(B):
        k = min(P, neg_ratio * int(ref["npos"][b]))
        paths.append(selection_path(key[b], k))
    finite = torch.isfinite(conf).all(-1) if finite_rows is None else finite_rows
    fin = finite.numpy()
    r = reference_f64(loc, conf, ref, mined.numpy())
    # CE accuracy: the kernel's taps and ATen's fp32 CE within the same bound of the float64 CE
    bound = ce_bound(conf.numpy(), r["ce"])
    err = np.abs(ce_tap.double().numpy() - r["ce"])
    bad = fin & ~(err <= bound)
    assert not bad.any(), f"{int(bad.sum())} kernel CE values outside the bound; worst {(err - bound)[fin].max():.3e}"
    aerr = np.abs(ref["cce"].double().numpy() - r["ce"])
    assert not (fin & ~(aerr <= bound)).any(), "the ATen fp32 oracle is outside the CE bound"
    # the float64 mined set may differ only at the boundary: within twice the bound of the k-th key
    with np.errstate(invalid="ignore"):
        v64 = np.where(pos.numpy(), 0.0, r["ce"])
    for b in range(B):
        k = min(P, neg_ratio * int(ref["npos"][b]))
        if not fin[b].all() or k == 0:
            continue
        m64 = O.mine_hard_negatives(torch.from_numpy(v64[b:b + 1]), pos[b:b + 1], neg_ratio)[0].numpy()
        diff = m64 ^ mined[b].numpy()
        if diff.any():
            kth = np.sort(v64[b])[::-1][k - 1]
            j = int(np.argmin(np.abs(v64[b] - kth)))
            assert (np.abs(v64[b][diff] - kth) <= 2 * bound[b, j] + 2 * bound[b][diff]).all(), \
                f"image {b}: float64 mined set differs away from the boundary"
    # sums and losses
    sel = pos.numpy() | mined.numpy()
    tap_sum = ce_tap.double().numpy()[sel].sum()
    s1 = float(o["sums"][1])
    if np.isfinite(tap_sum):
        assert abs(s1 - tap_sum) <= 1e-12 * abs(tap_sum), f"sums[1] {s1!r} vs float64 sum of the taps {tap_sum!r}"
    else:
        assert (np.isnan(s1) and np.isnan(tap_sum)) or s1 == tap_sum
    l1 = r["sums"][0]
    budget = EPS * (0.5 * np.abs(r["dl"]) + 4.0 * np.abs(r["tgt"])).sum() + 1e-12 * l1
    assert abs(float(o["sums"][0]) - l1) <= budget, (float(o["sums"][0]), l1, budget)
    N = r["N"]
    assert o["losses"][0].item() == float(np.float32(float(o["sums"][0]) / (4.0 * N)))
    with np.errstate(invalid="ignore"):
        q1 = np.float32(s1 / N)
    assert same_bits(o["losses"][1:2], torch.tensor([q1])), "conf loss is not the fp32 quotient of sums[1]"
    # gradients row by row, finite rows; a row outside the selection must be exactly zero
    check_grads(o, r, fin, pos.numpy(), loc)
    return paths, r, ref, mined


def check_grads(o, r, fin, pos, loc):
    gc = o["grad_conf"].double().numpy()
    err = np.abs(gc - r["grad_conf"])
    bad = fin[..., None] & ~(err <= r["grad_bound"])
    if bad.any():
        b, j, q = np.argwhere(bad)[0]
        raise AssertionError(f"grad_conf: {int(bad.any(-1).sum())} rows outside the bound, e.g. image {b} row {j} class {q}: "
                             f"{gc[b, j, q]!r} vs {r['grad_conf'][b, j, q]!r} (bound {r['grad_bound'][b, j, q]:.3e})")
    N = r["N"]
    gs = float(np.float32(1.0) / (np.float32(4.0) * np.float32(N)))
    gl = o["grad_loc"].double().numpy()
    want = np.zeros_like(gl)
    want[pos] = np.sign(r["dl"]) * gs
    near = np.zeros(pos.shape + (4,), bool)
    near[pos] = np.abs(r["dl"]) <= 8 * EPS * np.abs(r["tgt"])      # target one ulp away: the sign may differ
    assert ((gl == want) | near).all(), "grad_loc differs from sign(loc - target) / 4N"


def grad_check_sees_a_zeroed_row(o, r, fin, pos, loc, mined):
    """The gradient check must be able to fail: zero one mined row (a zero-CE one where there is one)."""
    gc = o["grad_conf"].clone()
    rows = np.argwhere(mined & fin)
    if rows.size == 0:
        return
    zero = [(b, j) for b, j in rows if float(o["ce"][b, j]) == 0.0]
    b, j = (zero or rows.tolist())[0]
    gc[b, j] = 0.0
    with pytest.raises(AssertionError):
        check_grads(dict(o, grad_conf=gc), r, fin, pos, loc)


# ----------------------------------------------------------------------------------------------------------- CPU tests
def test_float64_reference_against_fp32_oracle():
    """The float64 reference reproduces the fp32 oracle's losses and gradients on ordinary and trained logits."""
    for name in ("margin_17", "margin_40"):
        pri, loc, conf, tb, tc = case_inputs(name)
        ref = O.multibox_loss(loc, conf, tb, tc, pri)
        r = reference_f64(loc, conf, ref, ref["mined"].numpy())
        N = r["N"]
        assert abs(r["sums"][0] / (4 * N) - ref["loc_loss"].item()) <= 1e-6 * ref["loc_loss"].item()
        assert abs(r["sums"][1] / N - ref["conf_loss"].item()) <= 1e-5 * ref["conf_loss"].item()
        assert (np.abs(ref["cce"].double().numpy() - r["ce"]) <= ce_bound(conf.numpy(), r["ce"])).all()
        gl, gc = O.multibox_grads(loc, conf, ref)
        assert (np.abs(gc.double().numpy() - r["grad_conf"]) <= r["grad_bound"]).all()
        assert np.array_equal(gl.double().numpy(), r["grad_loc"].astype(np.float32).astype(np.float64))


@pytest.mark.parametrize("name", CASES)
def test_trained_generator_properties(name):
    """The families do what they are for: from margin 17 up, more rows of exactly zero CE per image than k; the
    margin-40 batch has images that select at T == 0 on the radix path."""
    pri, loc, conf, tb, tc = case_inputs(name)
    ref = O.multibox_loss(loc, conf, tb, tc, pri)
    pos = ref["pos"].numpy()
    zero = ((ref["cce"].numpy() == 0) & ~pos).sum(1)
    k = 3 * ref["npos"].numpy()
    if name in ("margin_17", "margin_25", "margin_40", "scaled", "bf16"):
        assert (zero > k).all(), (zero, k)
    key = keys_of(ref["cce"].numpy(), pos)
    paths = [selection_path(key[b], int(k[b])) for b in range(len(tb))]
    if name == "margin_40":
        assert any(p == ("radix", 0) for p in paths), paths
    if name == "margin_10":
        assert any(p[0] == "fast" for p in paths), paths
    if name == "bf16":
        v = ref["cce"].numpy()[~pos]
        assert v.size - np.unique(v).size > 1000, "bf16 logits should give thousands of exact CE ties"


def zero_boundary_inputs():
    """Images whose k-th key is 0 on the FAST path: a 1024-prior table, a few hundred negatives of exactly zero CE at
    random priors, 40 negatives with CE ~ 1e-6 (in the boundary bin, above the zeros), every other negative at CE
    ~ 0.1-5, and neg_ratio chosen so that k reaches npos + 20 ranks into the zero keys - positives, which rank with
    value 0, take some of those ranks (ties to the lower prior index)."""
    pri = H.priors()[5000:6024].contiguous()
    P = pri.shape[0]
    B = 2
    gb, gc = synth.make_gt(811, B, 6, 6)
    tb = [torch.from_numpy(b) for b in gb]
    tc = [torch.from_numpy(c) for c in gc]
    cls = class_map(pri, tb, tc)
    rng = np.random.Generator(np.random.PCG64(812))
    conf = trained_conf(813, cls, 2.0, hard=0.0, mis=0.0).numpy()
    npos = (cls != BG).sum(1)
    neg_ratio = int(np.ceil((P - 300) / npos.min()))
    for b in range(B):
        negs = np.nonzero(cls[b] == BG)[0]
        k = min(P, neg_ratio * int(npos[b]))
        n_above = k - int(npos[b]) - 20                 # negatives with CE > 0; the remaining ranks go to zero keys
        low = rng.choice(negs, negs.size - n_above + 40, replace=False)
        zero, tiny = low[40:], low[:40]
        conf[b, low, :BG] = rng.standard_normal((low.size, BG), dtype=np.float32)
        conf[b, zero, BG] = np.float32(60.0)
        conf[b, tiny, BG] = np.float32(16.0)
    return pri, torch.from_numpy(synth.make_head(814, B, P)[0]), torch.from_numpy(conf), tb, tc, neg_ratio


def test_zero_boundary_inputs_take_the_fast_zero_bin():
    pri, loc, conf, tb, tc, neg_ratio = zero_boundary_inputs()
    ref = O.multibox_loss(loc, conf, tb, tc, pri, ratio=neg_ratio)
    pos = ref["pos"].numpy()
    key = keys_of(ref["cce"].numpy(), pos)
    for b in range(len(tb)):
        k = min(pri.shape[0], neg_ratio * int(ref["npos"][b]))
        path = selection_path(key[b], k)
        assert path[0] == "fast" and path[1] == 0, path
        assert kernel_rank_positives_in(key[b], pos[b], ref["mined"][b].numpy(), k)


def natural_key_max(pri, conf, tb, tc, b):
    """The largest mining key of image b before the forced match (what the fused finaliser's kernel scales by)."""
    iou = O.iou_matrix(tb[b].view(-1, 4), O.cxcywh_to_xyxy(pri))
    ov, obj = iou.max(dim=0)
    natural_pos = (ov >= 0.5) & (tc[b][obj] != BG)
    ce_bg = O.cross_entropy_rows(conf[b:b + 1], torch.full((1, pri.shape[0]), BG))[0]
    return float(ce_bg[~natural_pos].max()), natural_pos


BG_PRIOR = 3001          # a level-0 prior in the middle of the image (no other prior has its box)


def bg_gt_inputs(kind):
    """A natural positive forced to the background: image 0 holds two gts with the box of prior BG_PRIOR, class 5 then
    class C-1.  The first is the prior's natural match (T1: lowest gt index), the second wins the forced match (T3:
    highest gt index), so the prior becomes a negative whose key rises from 0 to its CE.
      mild:    N(0,1) logits; the prior's background CE is set to 1.00073 x the image's largest natural key, so its
               fast-path bin is 2048 when the histogram is scaled by the natural keys alone.
      trained: margin-25 logits; the prior's background CE is ~20, its bin (scaled by the natural keys) past 8192.  Image 1 holds a
               background-labelled gt that is the natural best match of some priors; image 2 a forced prior whose
               conf row holds a NaN."""
    pri = H.priors()
    P = pri.shape[0]
    B = 2 if kind == "mild" else 3
    gb, gc = synth.make_gt(900, B, 3, 6)
    tb = [torch.from_numpy(b) for b in gb]
    tc = [torch.from_numpy(c) for c in gc]
    box = O.cxcywh_to_xyxy(pri[BG_PRIOR:BG_PRIOR + 1])
    tb[0] = torch.cat([box, box, tb[0]])
    tc[0] = torch.cat([torch.tensor([5.0, float(BG)]), tc[0]])
    if kind == "trained":
        tb[2] = torch.cat([box, box, tb[2]])
        tc[2] = torch.cat([torch.tensor([7.0, float(BG)]), tc[2]])
        tb[1][0] = O.cxcywh_to_xyxy(pri[7000:7001])[0]     # gt 0 of image 1: background-labelled, the box of a prior
        tc[1][0] = float(BG)
    loc = torch.from_numpy(synth.make_head(901, B, P)[0])
    if kind == "mild":
        conf = torch.from_numpy(synth.make_head(902, B, P)[1])
        vmax, _ = natural_key_max(pri, conf, tb, tc, 0)
        target = 1.00073 * vmax
        a = target - np.log(20.0)
        for _ in range(50):
            a = target - np.log(20.0 + np.exp(-a))
        conf[0, BG_PRIOR] = 0.0
        conf[0, BG_PRIOR, BG] = float(np.float32(-a))
    else:
        cls = class_map(pri, tb, tc)
        cls[0, BG_PRIOR] = 5                       # confidently its natural class: background CE ~ 25
        cls[2, BG_PRIOR] = 7
        conf = trained_conf(903, cls, 25.0)
        conf[2, BG_PRIOR, 3] = float("nan")
    return pri, loc, conf, tb, tc


def test_background_gt_mild_case_lands_in_bin_2048():
    pri, loc, conf, tb, tc = bg_gt_inputs("mild")
    vmax, natural_pos = natural_key_max(pri, conf, tb, tc, 0)
    assert bool(natural_pos[BG_PRIOR])
    ref = O.multibox_loss(loc, conf, tb, tc, pri)
    assert int(ref["cls"][0, BG_PRIOR]) == BG, "the forced match must make the prior a negative"
    key = np.float32(ref["cce"][0, BG_PRIOR].item())
    scale = np.float32(2047.0) / np.float32(vmax)
    assert int(np.float32(key * scale)) == 2048
    k = 3 * int(ref["npos"][0])
    nat = keys_of(ref["cce"][0].numpy(), natural_pos.numpy())
    assert selection_path(nat, k)[0] == "fast"


def test_background_gt_trained_inputs():
    pri, loc, conf, tb, tc = bg_gt_inputs("trained")
    ref = O.multibox_loss(loc, conf, tb, tc, pri)
    assert int(ref["cls"][0, BG_PRIOR]) == BG and int(ref["cls"][2, BG_PRIOR]) == BG
    vmax, natural_pos = natural_key_max(pri, conf, tb, tc, 0)
    assert bool(natural_pos[BG_PRIOR])
    assert ref["cce"][0, BG_PRIOR].item() * 2047 / vmax > 4 * 2048, "the key's bin must lie far past the histogram"
    assert torch.isnan(ref["cce"][2, BG_PRIOR])
    iou = O.iou_matrix(tb[1][:1], O.cxcywh_to_xyxy(pri))[0]
    assert bool(((iou >= 0.5) & (ref["cls"][1] == BG)).any()), "the background gt wins no prior"


# ----------------------------------------------------------------------------------------------------------- GPU tests
def _check_case(pri, loc, conf, tb, tc, neg_ratio=3, pos_iou=0.5, **kw):
    outs = run_routes(pri, loc, conf, tb, tc, neg_ratio, pos_iou, **kw)
    assert_routes_agree(outs)
    paths = None
    for name in ("flat", "three"):
        paths, r, ref, mined = check_against_references(pri, loc, conf, tb, tc, outs[name], neg_ratio, pos_iou)
    fin = torch.isfinite(conf).all(-1).numpy()
    grad_check_sees_a_zeroed_row(outs["flat"], r, fin, ref["pos"].numpy(), loc, mined.numpy())
    return outs, paths, ref


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_trained_case_all_routes(name):
    pri, loc, conf, tb, tc = case_inputs(name)
    _, paths, _ = _check_case(pri, loc, conf, tb, tc)
    if name == "margin_40":
        assert any(p == ("radix", 0) for p in paths), paths


@pytest.mark.gpu
def test_zero_boundary_fast_path_ranks_positives():
    pri, loc, conf, tb, tc, neg_ratio = zero_boundary_inputs()
    outs, paths, ref = _check_case(pri, loc, conf, tb, tc, neg_ratio=neg_ratio)
    pos = ref["pos"].numpy()
    mined = H.unpack_mask(outs["flat"]["mined_mask"], pri.shape[0]).numpy()
    key = keys_of(outs["flat"]["ce"].numpy(), pos)
    for b in range(len(tb)):
        assert paths[b][0] == "fast" and paths[b][1] == 0, paths[b]
        assert kernel_rank_positives_in(key[b], pos[b], mined[b], 0)


@pytest.mark.gpu
@pytest.mark.parametrize("neg_ratio,pos_iou", [(0, 0.5), (1, 0.5), (3, 0.35), (3, 0.7)])
def test_trained_hyperparameters(neg_ratio, pos_iou):
    pri, loc, conf, tb, tc = case_inputs("margin_17")
    _check_case(pri, loc, conf, tb, tc, neg_ratio=neg_ratio, pos_iou=pos_iou)


@pytest.mark.gpu
def test_background_gt_mild():
    """The forced background prior's key is just above the natural keys: it must be ranked like any other key (not k + 1
    mined negatives in the image)."""
    pri, loc, conf, tb, tc = bg_gt_inputs("mild")
    outs, _, ref = _check_case(pri, loc, conf, tb, tc)
    mined = H.unpack_mask(outs["flat"]["mined_mask"], pri.shape[0])
    assert int(mined[0].sum()) == 3 * int(ref["npos"][0])


@pytest.mark.gpu
def test_background_gt_trained():
    """Forced background prior with a key far above the natural keys, a background gt that is the natural best match
    of some priors, and a forced prior whose conf holds NaN (its key ranks above every finite key)."""
    pri, loc, conf, tb, tc = bg_gt_inputs("trained")
    outs, paths, ref = _check_case(pri, loc, conf, tb, tc)
    mined = H.unpack_mask(outs["flat"]["mined_mask"], pri.shape[0])
    assert bool(mined[0, BG_PRIOR]) and bool(mined[2, BG_PRIOR])
    assert np.isnan(float(outs["flat"]["sums"][1])) and np.isnan(float(ref["conf_loss"]))
    assert paths[2][0] == "radix"


@pytest.mark.gpu
@pytest.mark.parametrize("neg_ratio", [3, 0])
def test_nonfinite_background_logits(neg_ratio):
    """NaN, +inf and -inf in the background logit of a few negative rows: ranked NaN > +inf > finite (torch.sort's
    order); the conf loss is non-finite exactly where the oracle's is; the finite rows' gradients are unchanged."""
    pri, loc, conf, tb, tc = case_inputs("margin_25", seed=3)
    ref0 = O.multibox_loss(loc, conf, tb, tc, pri)
    rng = np.random.Generator(np.random.PCG64(950))
    for b in range(conf.shape[0]):
        negs = np.nonzero(~ref0["pos"][b].numpy())[0]
        rows = rng.choice(negs, 6, replace=False)
        for j, v in zip(rows, (float("nan"), float("inf"), float("-inf")) * 2):
            conf[b, j, BG] = v
    outs, _, ref = _check_case(pri, loc, conf, tb, tc, neg_ratio=neg_ratio)
    got = outs["flat"]["losses"]
    assert bool(torch.isfinite(got[0]))
    assert np.isfinite(got[1].item()) == np.isfinite(ref["conf_loss"].item())
    assert np.isnan(got[1].item()) == np.isnan(ref["conf_loss"].item())
    if neg_ratio:
        assert np.isnan(got[1].item())


@pytest.mark.gpu
def test_fallback_batch_300():
    """B = 300 takes the three-kernel route by itself: the images of a trained batch of 4, repeated, give the same taps
    and mined sets as the batch of 4, the mined set follows the rule on the taps, sums[1] is their float64 sum."""
    from objectdetection_ssd_b200.head import PackedGT
    from objectdetection_ssd_b200 import _lib
    pri, loc, conf, tb, tc = case_inputs("margin_25")
    head = _head(pri)
    small = head.loss(loc.cuda(), conf.cuda(), PackedGT(tb, tc, head.dev), with_grads=True, taps=True)
    reps = 75
    L, Cf = loc.repeat(reps, 1, 1).cuda(), conf.repeat(reps, 1, 1).cuda()
    n0 = _lib.launch_count()
    big = head.loss(L, Cf, PackedGT(tb * reps, tc * reps, head.dev), with_grads=True, taps=True)
    torch.cuda.synchronize()
    assert _lib.launch_count() - n0 >= 3, "B = 300 should take the three-kernel route"
    P = pri.shape[0]
    assert torch.equal(big["ce"].cpu(), small["ce"].cpu().repeat(reps, 1))
    assert torch.equal(big["mined_mask"].cpu(), small["mined_mask"].cpu().repeat(reps, 1))
    pos = big["cls_u8"].cpu() != BG
    ce = big["ce"].cpu()
    mined = H.unpack_mask(big["mined_mask"], P)
    assert torch.equal(mined, O.mine_hard_negatives(ce, pos, 3))
    s = ce.double().numpy()[(pos | mined).numpy()].sum()
    assert abs(float(big["sums"][1]) - s) <= 1e-12 * s


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_autograd_low_precision_inputs(dtype):
    """multibox_loss with bf16 / fp16 loc and conf: losses equal the fp32 route on the upcast inputs bit for bit, the
    gradients come back in the input dtype as the fp32 gradients cast to it; a non-contiguous conf view gives the same;
    backward on one loss alone leaves a zero gradient on the other input."""
    from objectdetection_ssd_b200.head import PackedGT, multibox_loss
    pri, loc, conf, tb, tc = case_inputs("margin_17")
    head = _head(pri)
    l16 = loc.to(dtype).cuda().requires_grad_(True)
    c16 = conf.to(dtype).cuda().requires_grad_(True)
    a, b = multibox_loss(head, l16, c16, tb, tc)
    (a + b).backward()
    ref = head.loss(l16.detach().float(), c16.detach().float(), PackedGT(tb, tc, head.dev), with_grads=True)
    torch.cuda.synchronize()
    assert same_bits(torch.stack([a.detach(), b.detach()]).cpu(), ref["losses"].cpu())
    assert l16.grad.dtype == dtype and c16.grad.dtype == dtype
    assert torch.equal(l16.grad, ref["grad_loc"].to(dtype)) and torch.equal(c16.grad, ref["grad_conf"].to(dtype))
    # a non-contiguous conf: a [B, C, P] tensor seen through a transpose
    base = conf.to(dtype).cuda().transpose(1, 2).contiguous().requires_grad_(True)
    view = base.transpose(1, 2)
    assert not view.is_contiguous()
    a2, b2 = multibox_loss(head, l16.detach(), view, tb, tc)
    b2.backward()
    assert same_bits(torch.stack([a2.detach(), b2.detach()]).cpu(), ref["losses"].cpu())
    assert torch.equal(base.grad.transpose(1, 2), ref["grad_conf"].to(dtype))
    # backward on the loc loss alone: the conf input gets a zero gradient
    l3 = loc.to(dtype).cuda().requires_grad_(True)
    c3 = conf.to(dtype).cuda().requires_grad_(True)
    a3, _ = multibox_loss(head, l3, c3, tb, tc)
    a3.backward()
    assert torch.equal(l3.grad, ref["grad_loc"].to(dtype)) and bool((c3.grad == 0).all())
    l4 = loc.to(dtype).cuda().requires_grad_(True)
    c4 = conf.to(dtype).cuda().requires_grad_(True)
    _, b4 = multibox_loss(head, l4, c4, tb, tc)
    b4.backward()
    assert torch.equal(c4.grad, ref["grad_conf"].to(dtype)) and bool((l4.grad == 0).all())
