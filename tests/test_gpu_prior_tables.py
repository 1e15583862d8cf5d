"""GPU: the training step and detect on prior tables in any order, against the oracle and against each other.

Every other GPU test runs on tables in SSD order (level, row, column, ratio): consecutive priors are spatial neighbours
with repeating areas, and the kernels use that order to skip work - the per-warp bounding-box skip of the match, the
``owns_p0`` exception of the warp that holds prior 0 (rule T2), the seeded area cull of the fused match, and the sampled
score floor of detect.  A user may hand the drop-in any table, so the results must not depend on that order.  The
tables here break it on purpose:

    perm        SSD300 rows under a random permutation: every warp's priors cover the whole image
    area        SSD300 sorted by the kernels' own fp32 area (stable): equal areas per warp, positions scattered, so
                the area cull is the only skip that fires
    rev         SSD300 reversed: prior 0 is a prior of the 1x1 level
    dup         SSD300 with 100 rows overwritten by exact copies of rows thousands of indices earlier: best-prior ties
                between warps, tiles and CTAs, which must go to the lower index (T2)
    rand        5003 random boxes, centres U(-0.1, 1.1), sides log-uniform in [0.01, 1.2], not clamped: an odd prior
                count (plain-load paths), boxes beyond the image, untidy values for the host corner conversion
    ssd512perm  SSD512 permuted, 100 gts per image: the stress shape, where the cull is on by default

Every prior has a positive area.  The oracle's tie rules are stated on prior indices, so it stays the reference on a
permuted table.
"""
import functools
import os
from collections import namedtuple

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from objectdetection_ssd_b200 import synth
from objectdetection_ssd_b200.priors import cxcywh_to_xyxy_host
from oracle import ssd_oracle as O
from tests import helpers as H
from tests.test_gpu_detect import _check_exact, _oracle_stage
from tests.test_gpu_detect_shortlist import _route, _same
from tests.test_gpu_loss import _check_loss, _check_match

pytestmark = pytest.mark.gpu

TABLES = ("perm", "area", "rev", "dup", "rand", "ssd512perm")
PERMUTED = ("perm", "area", "rev")
DETECT_TABLES = ("perm", "rev", "rand")
FAR_GT = [2.0, 2.0, 2.1, 2.1]            # overlaps no prior of any table here: T2 sends it to prior 0
Table = namedtuple("Table", "pri pi pairs")   # pri == base[pi] for the permuted tables; pairs (src, dst) of `dup`


def _area(pri):
    """The kernels' box_area of every prior: (x2 - x1) * (y2 - y1) in fp32 on the host corner form."""
    xy = cxcywh_to_xyxy_host(pri)
    return (xy[:, 2] - xy[:, 0]) * (xy[:, 3] - xy[:, 1])


@functools.lru_cache(maxsize=None)
def _table(name):
    g = torch.Generator().manual_seed(7100 + TABLES.index(name))
    pi, pairs = None, None
    if name in ("perm", "area", "rev", "ssd512perm"):
        base = H.priors("ssd512" if name == "ssd512perm" else "ssd300")
        P = base.shape[0]
        if name == "area":
            pi = torch.from_numpy(np.argsort(_area(base).numpy(), kind="stable"))
        elif name == "rev":
            pi = torch.arange(P - 1, -1, -1)
        else:
            pi = torch.randperm(P, generator=g)
        pri = base[pi]
    elif name == "dup":
        pri = H.priors().clone()
        P = pri.shape[0]
        dst = (torch.randperm(P - 3000, generator=g)[:100] + 3000).sort().values
        src = (torch.rand(100, generator=g) * (dst - 2000).double()).long()
        src[torch.isin(src, dst)] -= 1                           # copy from rows that keep their own value
        assert not torch.isin(src, dst).any() and ((dst - src) >= 2000).all()
        pri[dst] = pri[src]
        pairs = list(zip(src.tolist(), dst.tolist()))
    elif name == "rand":
        P = 5003
        c = -0.1 + 1.2 * torch.rand(P, 2, generator=g, dtype=torch.float64)
        s = torch.exp(np.log(0.01) + (np.log(1.2) - np.log(0.01)) * torch.rand(P, 2, generator=g, dtype=torch.float64))
        pri = torch.cat([c, s], 1).float()
    else:
        raise ValueError(name)
    pri = pri.contiguous()
    assert (_area(pri) > 0).all()
    return Table(pri, pi, pairs)


@functools.lru_cache(maxsize=None)
def _head(name):
    from objectdetection_ssd_b200.head import MultiboxHead
    return MultiboxHead(_table(name).pri, "cuda")


def _packed(tb, tc, head):
    from objectdetection_ssd_b200.head import PackedGT
    return PackedGT(tb, tc, head.dev)


def _gts(name, seed, B, dense):
    """Ragged gts for table ``name``: 1-10 (``dense``: 60-100; ssd512perm always 100) boxes per image, plus at the end
    of image 0 a gt that overlaps no prior (T2 -> prior 0) and in image 1 its first gt twice more (T3).  On ``dup``
    every image starts with the corner forms of 5 duplicated priors (_dup_pick): IoU 1 with a row and with its copy
    thousands of rows later."""
    t = _table(name)
    lo, hi = (100, 100) if name == "ssd512perm" else ((60, 100) if dense else (1, 10))
    gb, gc = synth.make_gt(seed, B, lo, hi)
    tb = [torch.from_numpy(b).clone() for b in gb]
    tc = [torch.from_numpy(c).clone() for c in gc]
    if t.pairs is not None:
        xy = cxcywh_to_xyxy_host(t.pri)
        for b in range(B):
            tb[b] = torch.cat([xy[[d for _, d in _dup_pick(t, b)]], tb[b]])
            tc[b] = torch.cat([torch.arange(5, dtype=torch.float32) + b % 3, tc[b]])
    tb[0] = torch.cat([tb[0], torch.tensor([FAR_GT])])
    tc[0] = torch.cat([tc[0], torch.tensor([11.0])])
    if B > 1:
        tb[1] = torch.cat([tb[1], tb[1][:1].repeat(2, 1)])
        tc[1] = torch.cat([tc[1], torch.tensor([4.0, 9.0])])
    return tb, tc


def _dup_pick(t, b):
    """The (source, copy) pairs of `dup` whose box image b holds as its first 5 gts."""
    return [t.pairs[(5 * b + 7 * j) % len(t.pairs)] for j in range(5)]


def _inputs(name, seed, B, dense):
    P = _table(name).pri.shape[0]
    loc, conf = synth.make_head(seed, B, P)
    tb, tc = _gts(name, seed, B, dense)
    return torch.from_numpy(loc), torch.from_numpy(conf), tb, tc


class _cull:
    """SSDHEAD_MATCH_CULL_MIN for the duration of a block: "1" forces the seeded cull on, a value above any average gt
    count forces it off."""

    def __init__(self, on):
        self.v = "1" if on else "1000000"

    def __enter__(self):
        self.old = os.environ.get("SSDHEAD_MATCH_CULL_MIN")
        os.environ["SSDHEAD_MATCH_CULL_MIN"] = self.v

    def __exit__(self, *a):
        if self.old is None:
            os.environ.pop("SSDHEAD_MATCH_CULL_MIN", None)
        else:
            os.environ["SSDHEAD_MATCH_CULL_MIN"] = self.old


def _assert_same_step(a, b, n, what):
    """Two training-step outputs (head.loss / loss_levels dicts) hold the same bits."""
    assert torch.equal(a["cls_u8"], b["cls_u8"]), f"{what}: class map"
    assert torch.equal(a["best_prior"][:n], b["best_prior"][:n]), f"{what}: best prior per gt"
    assert torch.equal(a["npos"], b["npos"]), f"{what}: positive counts"
    assert torch.equal(a["sums"], b["sums"]) and torch.equal(a["losses"], b["losses"]), f"{what}: loss sums"
    ga, gb = a["grad_loc"], b["grad_loc"]
    ca, cb = a["grad_conf"], b["grad_conf"]
    if isinstance(ga, list):
        ga, ca = torch.cat(ga, 1), torch.cat(ca, 1)
    assert torch.equal(ga, gb), f"{what}: grad_loc"
    assert torch.equal(ca, cb), f"{what}: grad_conf"


# ---------------------------------------------------------------------------------------------------------------------
# 1. the standalone match, exact

@pytest.mark.parametrize("name", TABLES)
def test_match_exact_on_every_table(name):
    """ssdhead_match against the oracle: class map, object map, best prior per gt (T2, including the gt that overlaps
    nothing and the duplicated priors of `dup`), positives - for ordinary and dense batches."""
    t = _table(name)
    head = _head(name)
    for seed, B, dense in ((11, 6, False), (12, 3, True)):
        tb, tc = _gts(name, seed, B, dense)
        gt, m, ref = _check_match(head, t.pri, tb, tc)
        assert int(m["best_prior"][tb[0].shape[0] - 1]) == 0, "a gt that overlaps no prior goes to prior 0 (T2)"
        if t.pairs is not None:
            bp = m["best_prior"].cpu()
            for b in range(B):                                   # a duplicated prior's box goes to the earlier copy
                for j, (src, dst) in enumerate(_dup_pick(t, b)):
                    assert int(bp[gt.off_host[b] + j]) == src, (b, j, int(bp[gt.off_host[b] + j]), src, dst)


# ---------------------------------------------------------------------------------------------------------------------
# 2. the training step against the oracle

@pytest.mark.parametrize("name", TABLES)
def test_step_against_the_oracle_on_every_table(name):
    """The flat two-kernel step with its taps (CE, mined mask, losses, both gradients) at the tolerances of
    test_gpu_loss._check_loss, and its fused match exactly equal to the oracle's."""
    pri = _table(name).pri
    B = 3 if name == "ssd512perm" else 12
    loc, conf, tb, tc = _inputs(name, 21, B, dense=False)
    out, ref = _check_loss(pri, loc, conf, tb, tc)
    n = sum(int(b.shape[0]) for b in tb)
    assert torch.equal(out["cls_u8"].cpu().long(), ref["cls"])
    assert torch.equal(out["best_prior"][:n].cpu().long(), ref["best_prior"])


# ---------------------------------------------------------------------------------------------------------------------
# 3. the seeded cull, forced on and forced off

@pytest.mark.parametrize("name", TABLES)
def test_cull_on_and_off_give_the_same_bits(name):
    """60-100 gts per image (100 on ssd512perm): the step with the seeded cull forced on and forced off gives the same
    class map, best priors, positives, sums, losses and gradients, and the class map and best priors are the
    oracle's."""
    head = _head(name)
    B = 3 if name == "ssd512perm" else 5
    loc, conf, tb, tc = _inputs(name, 31, B, dense=True)
    n = sum(int(b.shape[0]) for b in tb)
    outs = []
    for on in (True, False):
        with _cull(on):
            outs.append(head.loss(loc.cuda(), conf.cuda(), _packed(tb, tc, head), with_grads=True))
            torch.cuda.synchronize()
    _assert_same_step(outs[0], outs[1], n, f"{name}: cull on vs off")
    ref = O.match_batch(tb, tc, O.cxcywh_to_xyxy(_table(name).pri))
    assert torch.equal(outs[0]["cls_u8"].cpu().long(), ref["cls"])
    assert torch.equal(outs[0]["best_prior"][:n].cpu().long(), ref["best_prior"])


# ---------------------------------------------------------------------------------------------------------------------
# 4. every route of the step gives the flat step's bits

def _split(t, counts):
    out, s = [], 0
    for n in counts:
        out.append(t[:, s:s + n].contiguous())
        s += n
    return out


@pytest.mark.parametrize("name", TABLES)
def test_every_route_equals_the_flat_step(name):
    """Per-level step on a random level split, the three-kernel route on a standalone match, and the context's
    loss_dev, loss_dev_resident and loss_host (one chunk at these batch sizes) on a context created from the same
    table: the flat step's bits.  The context builds its corner table with its own host routine, so on `rand` this
    also pins that routine to the Python conversion."""
    from objectdetection_ssd_b200.ctx import SSDHeadContext
    head = _head(name)
    pri = _table(name).pri
    P = pri.shape[0]
    g = torch.Generator().manual_seed(41)
    for seed, B, dense in ((42, 12, False), (43, 8, True)):
        if name == "ssd512perm":
            B = 3
        loc, conf, tb, tc = _inputs(name, seed, B, dense)
        n = sum(int(b.shape[0]) for b in tb)
        l, c = loc.cuda(), conf.cuda()
        gt = _packed(tb, tc, head)
        flat = head.loss(l, c, gt, with_grads=True)
        L = int(torch.randint(2, 9, (1,), generator=g))
        cuts = sorted(set(torch.randint(1, P, (L - 1,), generator=g).tolist()))
        counts = [b - a for a, b in zip([0] + cuts, cuts + [P])]
        lv = head.loss_levels(_split(l, counts), _split(c, counts), gt, with_grads=True)
        torch.cuda.synchronize()
        _assert_same_step(lv, flat, n, f"{name} seed {seed}: per-level step, levels {counts}")
        m = head.match(gt)
        three = head.loss(l, c, gt, with_grads=True, match=m)
        torch.cuda.synchronize()
        _assert_same_step(three, flat, n, f"{name} seed {seed}: three-kernel route")

        gx, gcl, off = synth.pack_gt([b.numpy() for b in tb], [x.numpy() for x in tc])
        ctx = SSDHeadContext(pri.numpy(), max_batch=B, max_total_gt=max(n, 128 * B))
        try:
            d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
            tgx, tgc, toff = d(gx), d(gcl), d(off)
            st = torch.cuda.current_stream().cuda_stream
            for resident in (False, True):
                sums = torch.empty(2, dtype=torch.float64, device="cuda")
                losses = torch.empty(2, device="cuda")
                gl = torch.full_like(l, 7.0) if resident else torch.empty_like(l)
                gc = torch.full_like(c, -3.0) if resident else torch.empty_like(c)
                args = (l.data_ptr(), c.data_ptr(), tgx.data_ptr(), tgc.data_ptr(), toff.data_ptr(), B, n,
                        sums.data_ptr(), losses.data_ptr(), gl.data_ptr(), gc.data_ptr(), st)
                if resident:
                    ctx.loss_dev_resident(*args, fresh=True)
                else:
                    ctx.loss_dev(*args)
                torch.cuda.synchronize()
                what = f"{name} seed {seed}: context loss_dev{'_resident' if resident else ''}"
                assert torch.equal(sums, flat["sums"]) and torch.equal(losses, flat["losses"]), what
                assert torch.equal(gl, flat["grad_loc"]) and torch.equal(gc, flat["grad_conf"]), what
            hgl, hgc = np.empty_like(loc.numpy()), np.empty_like(conf.numpy())
            hl = ctx.loss_host(np.ascontiguousarray(loc.numpy()), np.ascontiguousarray(conf.numpy()), gx, gcl, off, hgl, hgc)
            fl = flat["losses"].cpu()
            assert hl == (float(fl[0]), float(fl[1])), f"{name} seed {seed}: context loss_host losses"
            assert torch.equal(torch.from_numpy(hgl), flat["grad_loc"].cpu()), f"{name} seed {seed}: loss_host grad_loc"
            assert torch.equal(torch.from_numpy(hgc), flat["grad_conf"].cpu()), f"{name} seed {seed}: loss_host grad_conf"
        finally:
            ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# 5. permutation equivariance

def _assert_no_ties(pri, tb):
    """Preconditions of the equivariance check: no two priors are equal, and every gt has one prior of strictly
    highest IoU, above 0 (a tie, or an all-zero row, is resolved by index, which the permutation changes)."""
    assert torch.unique(pri, dim=0).shape[0] == pri.shape[0], "duplicate priors"
    xy = O.cxcywh_to_xyxy(pri)
    for b, boxes in enumerate(tb):
        top = O.iou_matrix(boxes, xy).topk(2, dim=1).values
        assert (top[:, 0] > 0).all() and (top[:, 0] > top[:, 1]).all(), f"image {b}: a gt whose best prior is a tie"


def _assert_no_boundary_tie(out, P):
    """No CE at a mining boundary equals the CE just below it (T4 would resolve it by index)."""
    ce = out["ce"].cpu()
    pos = out["cls_u8"].cpu() != 20
    npos = out["npos"].cpu()
    for b in range(ce.shape[0]):
        v = ce[b].clone()
        v[pos[b]] = -1.0
        k = int(3 * npos[b])
        nneg = int((~pos[b]).sum())
        if 0 < k < nneg:
            s = torch.sort(v, descending=True).values
            assert s[k - 1] != s[k], f"image {b}: CE tie at the mining boundary"


def _untied_gts(seed, B, pri):
    """4-10 random gts per image, without the gts whose best prior is a tie (common: a gt that contains two priors of
    one area has the same IoU with both) or whose IoU is 0 with every prior."""
    gb, gc = synth.make_gt(seed, B, 4, 10)
    xy = O.cxcywh_to_xyxy(pri)
    tb, tc = [], []
    for b, c in zip(gb, gc):
        top = O.iou_matrix(torch.from_numpy(b), xy).topk(2, dim=1).values
        keep = (top[:, 0] > 0) & (top[:, 0] > top[:, 1])
        assert keep.any(), "an image without an untied gt: pick another seed"
        tb.append(torch.from_numpy(b)[keep].contiguous())
        tc.append(torch.from_numpy(c)[keep].contiguous())
    return tb, tc


@pytest.mark.parametrize("name", PERMUTED)
@pytest.mark.parametrize("B", [8, 256])
def test_step_is_permutation_equivariant(name, B):
    """On inputs without ties, the step on (pri[pi], loc[:, pi], conf[:, pi]) returns the step's per-row outputs on
    (pri, loc, conf) permuted by pi, bit for bit: class bytes, CE tap, mined mask, gradient rows; best priors map
    through pi.  The two loss sums are float64 sums of the same fp32 terms in another order: each is within
    (n - 1) 2^-53 of the exact sum of its n non-negative terms, so they differ by at most 2 n 2^-53 of the sum."""
    from objectdetection_ssd_b200.head import MultiboxHead
    t = _table(name)
    base = H.priors()
    P = base.shape[0]
    pi = t.pi
    assert torch.equal(t.pri, base[pi])
    loc, conf = (torch.from_numpy(a) for a in synth.make_head(5100 + B, B, P))
    tb, tc = _untied_gts(5100 + B, B, base)
    _assert_no_ties(base, tb)
    gt_b = _packed(tb, tc, _head(name))
    hb = MultiboxHead(base, "cuda")
    ob = hb.loss(loc.cuda(), conf.cuda(), gt_b, with_grads=True, taps=True)
    op = _head(name).loss(loc[:, pi].cuda(), conf[:, pi].cuda(), gt_b, with_grads=True, taps=True)
    torch.cuda.synchronize()
    _assert_no_boundary_tie(ob, P)
    n = gt_b.sumG
    pic = pi.cuda()
    assert torch.equal(op["cls_u8"], ob["cls_u8"][:, pic]), "class bytes"
    assert torch.equal(op["npos"], ob["npos"]), "positive counts"
    assert torch.equal(pic[op["best_prior"][:n].long()], ob["best_prior"][:n].long()), "best prior per gt"
    assert torch.equal(op["ce"], ob["ce"][:, pic]), "CE tap"
    mb, mp = H.unpack_mask(ob["mined_mask"], P), H.unpack_mask(op["mined_mask"], P)
    assert torch.equal(mp, mb[:, pi]), "mined mask"
    assert torch.equal(op["grad_loc"], ob["grad_loc"][:, pic]), "grad_loc rows"
    assert torch.equal(op["grad_conf"], ob["grad_conf"][:, pic]), "grad_conf rows"
    sp, sb = op["sums"].cpu(), ob["sums"].cpu()
    nterms = (4 * int(ob["npos"][-1]), int(ob["npos"][-1]) + int(mb.sum()))       # |loc - target| terms, CE terms
    for i in range(2):
        bound = 2.0 * nterms[i] * 2.0 ** -53 * float(sb[i])
        assert abs(float(sp[i]) - float(sb[i])) <= bound, (i, float(sp[i]), float(sb[i]), bound)
    lp, lb = op["losses"].cpu(), ob["losses"].cpu()
    assert torch.allclose(lp, lb, rtol=2.0 ** -22, atol=0), (lp, lb)     # one fp32 rounding of sums / count apart


# ---------------------------------------------------------------------------------------------------------------------
# 6. the margin of the seeded cull

def _iou_k(g, xy, pa):
    """The fused match's IoU of one gt box against priors, in the kernels' fp32 operation order."""
    ga = (g[2] - g[0]) * (g[3] - g[1])
    dx = np.minimum(g[2], xy[:, 2]) - np.maximum(g[0], xy[:, 0])
    dy = np.minimum(g[3], xy[:, 3]) - np.maximum(g[1], xy[:, 1])
    inter = dx * dy
    with np.errstate(all="ignore"):
        v = inter / ((ga + pa) - inter)
    return np.where((dx > 0) & (dy > 0), v, np.float32(0)).astype(np.float32)


def _ulp_steps(x, n):
    """The fp32 values from n ulps below x to n ulps above it."""
    down, up = [np.float32(x)], [np.float32(x)]
    for _ in range(n):
        down.append(np.nextafter(down[-1], np.float32(-np.inf)))
        up.append(np.nextafter(up[-1], np.float32(np.inf)))
    return np.array(down[:0:-1] + up, np.float32)


def _margin_gts(B, pos_iou=0.5):
    """Gts on the `area` table whose positivity is decided at the cull's rounding margin.

    Each gt is nested in a prior p with p's centre, so IoU(gt, p) = area(gt) / area(p) up to the rounding of the
    union.  p is no seed of match_seed_kernel (seeds are every 16th prior), the smallest area of p's warp in the
    streaming kernel's [B*P] rows equals area(p), so the warp's bound ub = area(gt) / area(p) rounded once, and a seed
    q outside p's warp overlaps the gt with IoU > pos_iou, so the gt's seed is above pos_iou and the cull compares ub
    with pos_iou itself.  In every image the exact ratios area(gt) / area(p) are pos_iou (1 + k 2^-23) for k = -4..4,
    to within half that step (fp32 boxes reach no closer), and one of them has an fp32 IoU with p of exactly pos_iou
    (T6: positive).  Returns (boxes, classes, info) - info rows (image, gt, p, target ratio, fp32 ratio = the cull's
    bound ub, fp32 IoU with p)."""
    f32 = np.float32
    pri = _table("area").pri
    P = pri.shape[0]
    xy = cxcywh_to_xyxy_host(pri).numpy()
    area = _area(pri).numpy()
    seeds = np.arange(0, P, 16)
    targets = [pos_iou * (1 + k * 2.0 ** -23) for k in range(-4, 5)]
    kinds = (lambda ub, iou: iou == pos_iou, lambda ub, iou: True)                    # a T6 box first, then any
    rng = np.random.Generator(np.random.PCG64(61))
    tb, tc, info = [], [], []
    for b in range(B):
        boxes, chosen, missing = [], [], list(range(len(targets)))
        for want in kinds:
            for p in rng.permutation(P):
                if not missing:
                    break
                r = b * P + p
                w0 = r // 32 * 32
                rows = np.arange(w0, min(w0 + 32, B * P)) % P
                pw, ph = xy[p, 2] - xy[p, 0], xy[p, 3] - xy[p, 1]
                if p % 16 == 0 or area[rows].min() != area[p] or pw > 0.35 or ph > 0.35 or p in chosen:
                    continue
                g = None
                for t in (0.95, 0.85, 0.75):
                    w = f32(t) * pw
                    h = f32(0.5) * area[p] / w
                    if h > f32(0.95) * ph:
                        continue
                    cand = np.array([pri[p, 0] - w / 2, pri[p, 1] - h / 2, pri[p, 0] + w / 2, pri[p, 1] + h / 2], f32)
                    v = _iou_k(cand, xy[seeds], area[seeds])
                    q = int(seeds[int(v.argmax())])
                    if v.max() > pos_iou * 1.001 and not (w0 <= b * P + q < w0 + 32):
                        g = cand
                        break
                if g is None:
                    continue
                # clear of the gts placed so far and of the priors deciding them: no other gt decides p's class
                if any(_iou_k(g, xy[[c]], area[[c]])[0] > 0.25 or _iou_k(o, xy[[p]], area[[p]])[0] > 0.25
                       for o, c in zip(boxes, chosen)):
                    continue
                # move the right and bottom edges by up to 24 ulps each, for a missing ratio and the wanted kind of box
                x2s, y2s = _ulp_steps(g[2], 24), _ulp_steps(g[3], 24)
                ga = (x2s[:, None] - g[0]) * (y2s[None, :] - g[1])
                exact = ga.astype(np.float64) / np.float64(area[p])
                found = None
                for k in missing:
                    for i, j in zip(*np.nonzero(np.abs(exact - targets[k]) <= pos_iou * 2.0 ** -24)):
                        cand = np.array([g[0], g[1], x2s[i], y2s[j]], f32)
                        ub = ga[i, j] / area[p]
                        iou = _iou_k(cand, xy[[p]], area[[p]])[0]
                        if cand[2] <= xy[p, 2] and cand[3] <= xy[p, 3] and want(ub, iou):
                            found = (k, cand, ub, iou)
                            break
                    if found:
                        break
                if found is None:
                    continue
                k, cand, ub, iou = found
                missing.remove(k)
                boxes.append(cand)
                chosen.append(p)
                info.append((b, len(boxes) - 1, int(p), targets[k], float(ub), float(iou)))
                if want is not kinds[-1]:
                    break                                        # one T6 box per image
        assert not missing, f"image {b}: no margin gt for the ratios {[targets[k] for k in missing]}"
        tb.append(torch.from_numpy(np.stack(boxes)))
        tc.append(torch.from_numpy(((np.arange(len(boxes)) * 3 + b) % 20).astype(np.float32)))
    return tb, tc, info


def test_cull_margin_on_the_area_table():
    """Gts whose IoU with the prior that decides them sits within a few ulps of pos_iou, on the table where the area
    cull is the only skip (see _margin_gts), among them gts whose IoU is exactly pos_iou (T6: positive).  With the cull
    forced on and off the step must give the same bits, and the oracle's class map and best priors.

    The cull's 1.00002 margin is not tight at these sizes: no box built here has an fp32 IoU of pos_iou or more while
    the rounded area ratio the cull bounds it with is below pos_iou (where the IoU rounds above the ratio, both stay on
    the same side), so a cull without the margin gives the same results.  This test pins the cull's exactness at
    ratios around pos_iou, not the margin's size."""
    name = "area"
    pri = _table(name).pri
    P = pri.shape[0]
    B = 4
    tb, tc, info = _margin_gts(B)
    # preconditions: the boxes really sit at the margin
    assert all(abs(ratio - 0.5) <= 5 * 2.0 ** -24 and abs(iou - 0.5) <= 5 * 2.0 ** -24 for *_, ratio, ub, iou in info)
    assert any(iou == 0.5 for *_, iou in info), "no gt at IoU == pos_iou (T6)"
    head = _head(name)
    ref = O.match_batch(tb, tc, O.cxcywh_to_xyxy(pri))
    for b, g, p, ratio, ub, iou in info:                          # the oracle agrees with the fp32 IoU: T6 at pos_iou
        assert bool(ref["pos"][b, p]) == (iou >= 0.5), (b, g, p, ratio, ub, iou)
    loc, conf = synth.make_head(62, B, P)
    loc, conf = torch.from_numpy(loc), torch.from_numpy(conf)
    n = sum(int(x.shape[0]) for x in tb)
    outs = []
    for on in (True, False):
        with _cull(on):
            outs.append(head.loss(loc.cuda(), conf.cuda(), _packed(tb, tc, head), with_grads=True))
            torch.cuda.synchronize()
    for o, what in zip(outs, ("cull on", "cull off")):
        cls = o["cls_u8"].cpu().long()
        bad = [row for row in info if int(cls[row[0], row[2]]) != int(ref["cls"][row[0], row[2]])]
        assert not bad, f"{what}: margin gts whose deciding prior has the wrong class: {bad}"
        assert torch.equal(cls, ref["cls"]), f"{what}: class map"
        assert torch.equal(o["best_prior"][:n].cpu().long(), ref["best_prior"]), f"{what}: best prior per gt"
    _assert_same_step(outs[0], outs[1], n, "margin gts: cull on vs off")
    _check_match(head, pri, tb, tc)


# ---------------------------------------------------------------------------------------------------------------------
# 7. detect

@pytest.mark.parametrize("name", DETECT_TABLES)
def test_detect_on_reordered_tables(name):
    """The fused detect on both routes against the oracle (boundary proofs of helpers.compare_detect_with_oracle), the
    stage-isolated path bit for bit against the oracle, the per-level entry on a random split equal to detect, and
    the two routes identical with the fallback count reported."""
    from objectdetection_ssd_b200.head import detect, detect_from_scores, detect_fallbacks, detect_levels
    head = _head(name)
    pri = _table(name).pri
    P = pri.shape[0]
    B = 4
    loc, conf = H.detect_inputs(81, B, P, bg_bias=6.0)
    outs = []
    for shortlist in (True, False):
        with _route(shortlist):
            outs.append(detect(head, loc, conf, 0.01, 0.45, 200))
            nfb = detect_fallbacks(head, B)
        torch.cuda.synchronize()
        assert 0 <= nfb <= B and (shortlist or nfb == 0), nfb
    _same(outs[0], outs[1])
    H.compare_detect_with_oracle(outs[0], loc, conf, pri, 0.01, 0.45, 200, range(B))

    boxes = torch.stack([O.decode(loc[i], pri) for i in range(B)])
    probs = F.softmax(conf, dim=2)
    ref = _oracle_stage(boxes, probs, 0.01, 0.45, 200)
    for shortlist in (True, False):
        with _route(shortlist):
            out = detect_from_scores(head, boxes, probs, 0.01, 0.45, 200)
        torch.cuda.synchronize()
        _check_exact(out, ref, 200, f"{name} shortlist={shortlist}")

    g = torch.Generator().manual_seed(82)
    L = int(torch.randint(2, 9, (1,), generator=g))
    cuts = sorted(set(torch.randint(1, P, (L - 1,), generator=g).tolist()))
    counts = [b - a for a, b in zip([0] + cuts, cuts + [P])]
    for shortlist in (True, False):
        with _route(shortlist):
            lv = detect_levels(head, _split(loc.cuda(), counts), _split(conf.cuda(), counts), 0.01, 0.45, 200)
        torch.cuda.synchronize()
        _same(lv, outs[0])
