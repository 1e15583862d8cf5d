"""GPU parity at the edges of the shapes the entry points accept.

The other GPU tests run well inside the supported shapes.  Past certain sizes the kernels change layout or code path,
so each limit is reached here - found from the library itself, not hard-coded - and checked against the CPU oracle:

- the loss at the largest prior count its mining kernel's shared-memory layout holds (``P_max``), on the dense, the
  sparse-row and the resident-gradient routes;
- gts per batch on both sides of the two 16-bit switches of the training step: the best-gt map (``sumG <= 65535``)
  and the seeded cull of the fused match (``sumG <= 65536``); above the first the fused finaliser walks every gt of
  the image for each positive row;
- detect at the largest prior count (``P = 512 x 256``), on both routes;
- detect at the largest accepted ``top_k`` (the kept list fills the sweep's shared memory), where most images of the
  short-list route need its fallback;
- ``get_map`` on the detections of a few hundred images (more than 65 536 of them) with adversarial additions.

One past each limit the call must be refused before anything is launched.  Run with ``-s`` to see the limits found and
the route each case took.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from objectdetection_ssd_b200 import synth
from oracle import ssd_oracle as O
from tests import helpers as H
from tests.test_gpu_detect import _check_exact, _clustered_inputs, _oracle_stage
from tests.test_gpu_detect_shortlist import _route, _same
from tests.test_gpu_loss import _check_loss, _check_match

pytestmark = pytest.mark.gpu

E_UNSUPPORTED = -2


def _head(pri):
    from objectdetection_ssd_b200.head import MultiboxHead
    return MultiboxHead(pri, "cuda")


def _launches():
    from objectdetection_ssd_b200 import _lib
    return _lib.launch_count()


def _prior_table(P, seed=0):
    """SSD512's 24 564 priors, then jittered copies of them up to ``P`` rows (a longer table is cut, so the tables of
    P and P - 1 share their first P - 1 rows)."""
    base = H.priors("ssd512")
    if P <= base.shape[0]:
        return base[:P].contiguous()
    g = torch.Generator().manual_seed(seed)
    n = P - base.shape[0]
    extra = base[torch.randint(0, base.shape[0], (n,), generator=g)].clone()
    extra[:, :2] += 0.01 * torch.randn(n, 2, generator=g)
    extra[:, 2:] *= torch.exp(0.05 * torch.randn(n, 2, generator=g))
    return torch.cat([base, extra]).contiguous()


# ---------------------------------------------------------------------------------------------------------------------
# 1. the loss at the largest supported prior count

@pytest.fixture(scope="module")
def p_max():
    """Largest P for which the loss workspace query is non-zero (no launch: a host-side size query)."""
    from objectdetection_ssd_b200 import _lib
    lib = _lib.load()
    ok = lambda P: lib.ssdhead_workspace_bytes(_lib.WS_LOSS, 4, P, 21, 0) > 0
    lo, hi = 8732, 1 << 17
    assert ok(lo) and not ok(hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if ok(mid) else (lo, mid)
    print(f"\n[limits] loss: P_max = {lo} priors")
    return lo


def _loss_inputs(P, seed):
    """Four images: 1..10 gts each, except image 1 with 150 (more than the 64 gts the mining kernel stages and the
    128 of the match kernels)."""
    B = 4
    gb, gc = synth.make_gt(seed, B, 1, 10)
    mb, mc = synth.make_gt(seed + 1, 1, 150, 150)
    gb[1], gc[1] = mb[0], mc[0]
    loc, conf = synth.make_head(seed + 2, B, P)
    return loc, conf, gb, gc


@pytest.mark.parametrize("below", [0, 1])
def test_loss_at_the_largest_prior_count(p_max, below):
    P = p_max - below
    pri = _prior_table(p_max)[:P].contiguous()
    loc, conf, gb, gc = _loss_inputs(P, 210)
    tb, tc = [torch.from_numpy(b) for b in gb], [torch.from_numpy(c) for c in gc]
    out, ref = _check_loss(pri, torch.from_numpy(loc), torch.from_numpy(conf), tb, tc)
    assert torch.equal(out["cls_u8"].cpu().long(), ref["cls"])
    assert torch.equal(out["best_prior"][:sum(len(b) for b in gb)].cpu().long(), ref["best_prior"])
    # positives sit near the end of the table too: the 16-bit row lists hold indices up to P - 1
    assert int(ref["pos"][:, P - 4096:].sum()) > 0
    print(f"[limits] loss at P = {P}: npos {ref['npos'].tolist()}, equal to the oracle")


def test_sparse_and_resident_routes_at_the_largest_prior_count(p_max):
    """The packed rows of the sparse route and the resident gradient tensors equal the dense step bit for bit."""
    from objectdetection_ssd_b200.ctx import SSDHeadContext, SparseRows, pinned_empty
    from objectdetection_ssd_b200.head import PackedGT
    P = p_max
    pri = _prior_table(P)
    loc, conf, gb, gc = _loss_inputs(P, 210)
    B = loc.shape[0]
    gx, gcl, off = synth.pack_gt(gb, gc)
    head = _head(pri)
    tb, tc = [torch.from_numpy(b) for b in gb], [torch.from_numpy(c) for c in gc]
    dense = head.loss(torch.from_numpy(loc).cuda(), torch.from_numpy(conf).cuda(), PackedGT(tb, tc, head.dev), with_grads=True)
    torch.cuda.synchronize()
    dgl, dgc = dense["grad_loc"].cpu().numpy(), dense["grad_conf"].cpu().numpy()
    ctx = SSDHeadContext(pri.numpy(), max_batch=B, max_total_gt=int(off[-1]))
    try:
        # sparse rows (host buffers in, packed rows out)
        hl, hc = pinned_empty(loc.shape), pinned_empty(conf.shape)
        hl[:] = loc
        hc[:] = conf
        rows = SparseRows(B, cap=P)
        rows.idx[...] = -1
        l1, l2 = ctx.loss_host_sparse(hl, hc, gx, gcl, off, rows)
        sgl, sgc = rows.scatter(P)
        assert np.array_equal(sgl, dgl) and np.array_equal(sgc, dgc), "sparse rows differ from the dense step"
        assert int(rows.idx[:, :].max()) >= P - 4096
        lo = dense["losses"].cpu()
        assert abs(l1 - lo[0].item()) <= 1e-6 * abs(lo[0].item()) and abs(l2 - lo[1].item()) <= 1e-6 * abs(lo[1].item())
        # resident gradient tensors: a first (fresh) step, then a step on other logits that retracts the first one's rows
        d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        tgx, tgc, toff = d(gx), d(gcl), d(off)
        st = torch.cuda.current_stream().cuda_stream
        gl_res = torch.full((B, P, 4), 7.0, device="cuda")
        gc_res = torch.full((B, P, 21), -3.0, device="cuda")
        sums = torch.empty(2, dtype=torch.float64, device="cuda")
        losses = torch.empty(2, device="cuda")
        sums_d = torch.empty(2, dtype=torch.float64, device="cuda")
        losses_d = torch.empty(2, device="cuda")
        _, conf2 = synth.make_head(219, B, P)
        for step, cf in enumerate((conf, conf2)):
            tl, tcf = d(loc), d(cf)
            ctx.loss_dev_resident(tl.data_ptr(), tcf.data_ptr(), tgx.data_ptr(), tgc.data_ptr(), toff.data_ptr(), B,
                                  int(off[-1]), sums.data_ptr(), losses.data_ptr(), gl_res.data_ptr(), gc_res.data_ptr(), st,
                                  fresh=step == 0)
            gl_d, gc_d = torch.empty_like(tl), torch.empty_like(tcf)
            ctx.loss_dev(tl.data_ptr(), tcf.data_ptr(), tgx.data_ptr(), tgc.data_ptr(), toff.data_ptr(), B, int(off[-1]),
                         sums_d.data_ptr(), losses_d.data_ptr(), gl_d.data_ptr(), gc_d.data_ptr(), st)
            torch.cuda.synchronize()
            assert torch.equal(losses, losses_d) and torch.equal(sums, sums_d), f"step {step}: losses"
            assert torch.equal(gc_res, gc_d), f"step {step}: resident grad_conf differs from the dense step"
            assert torch.equal(gl_res, gl_d), f"step {step}: resident grad_loc differs from the dense step"
            if step == 0:
                assert torch.equal(gc_d.cpu(), dense["grad_conf"].cpu()) and torch.equal(gl_d.cpu(), dense["grad_loc"].cpu())
                assert torch.equal(losses_d, dense["losses"])
    finally:
        ctx.close()
    print(f"[limits] loss at P = {P}: sparse rows and resident tensors equal the dense step")


def test_loss_one_prior_past_the_limit_is_refused_before_any_launch(p_max):
    from objectdetection_ssd_b200 import _lib
    from objectdetection_ssd_b200.head import PackedGT
    P = p_max + 1
    pri = _prior_table(P)
    loc, conf, gb, gc = _loss_inputs(P, 220)
    B = loc.shape[0]
    head = _head(pri)
    gt = PackedGT([torch.from_numpy(b) for b in gb], [torch.from_numpy(c) for c in gc], head.dev)
    l, c = torch.from_numpy(loc).cuda(), torch.from_numpy(conf).cuda()
    torch.cuda.synchronize()
    n0 = _launches()
    with pytest.raises(RuntimeError, match="unsupported shape"):
        head.loss(l, c, gt, with_grads=True)
    # the C entry point itself, given workspaces of the largest supported size: E_UNSUPPORTED
    lib = head.lib
    ws = torch.zeros(int(lib.ssdhead_workspace_bytes(_lib.WS_LOSS, B, p_max, 21, 0)), dtype=torch.uint8, device="cuda")
    wm = torch.zeros(int(lib.ssdhead_workspace_bytes(_lib.WS_MATCH, B, P, 21, gt.sumG)), dtype=torch.uint8, device="cuda")
    m = head._match_outputs(gt, False)
    sums = torch.empty(2, dtype=torch.float64, device="cuda")
    losses = torch.empty(2, device="cuda")
    gl, gcf = torch.empty_like(l), torch.empty_like(c)
    torch.cuda.synchronize()
    rc = lib.ssdhead_multibox_step(l.data_ptr(), c.data_ptr(), gt.boxes.data_ptr(), gt.classes.data_ptr(), gt.off.data_ptr(),
                                   head.pri_xyxy.data_ptr(), head.pri_cxcywh.data_ptr(), B, P, 21, gt.sumG, 3, 0.5,
                                   sums.data_ptr(), losses.data_ptr(), gl.data_ptr(), gcf.data_ptr(), m["cls_u8"].data_ptr(),
                                   m["best_prior"].data_ptr(), m["npos"].data_ptr(), None, None, ws.data_ptr(), ws.numel(),
                                   wm.data_ptr(), wm.numel(), torch.cuda.current_stream().cuda_stream)
    assert rc == E_UNSUPPORTED, rc
    assert _launches() == n0, "a refused call launched kernels"
    print(f"[limits] loss at P = {P}: refused (E_UNSUPPORTED), no launch")


# ---------------------------------------------------------------------------------------------------------------------
# 2. gts per batch across the 16-bit switches of the training step

OBJ_MAP_MAX = 65535      # the best-gt map of the streaming kernel holds a gt index in 16 bits
SEED_CAP = 65536         # gts the seeded cull of the fused match has seeds for


def _dense_gt_batch(sumG):
    """64 images of 1 024 gts (most priors positive), image 0 trimmed or extended so the batch holds ``sumG`` gts.
    Tiny, whole-image, duplicate and prior-identical gts on both sides of the 64 gts the mining kernel stages."""
    B = 64
    gb, gc = synth.make_gt(301, B, 1024, 1024)
    tb = [torch.from_numpy(b).clone() for b in gb]
    tc = [torch.from_numpy(c).clone() for c in gc]
    pri = H.priors()
    prior_box = torch.cat([pri[4000, :2] - pri[4000, 2:] / 2, pri[4000, :2] + pri[4000, 2:] / 2])
    tb[1][0] = torch.tensor([0.50, 0.50, 0.505, 0.505])         # tiny
    tb[1][1] = torch.tensor([0.0, 0.0, 1.0, 1.0])               # the whole image
    tb[1][3] = tb[1][2].clone()                                 # duplicates among the staged gts
    tb[2][700] = tb[2][100].clone()                             # duplicates past them (T2 / T3 ties)
    tb[3][900] = prior_box                                      # exactly a prior
    tb[4][1023] = torch.tensor([0.0, 0.0, 1.0, 1.0])
    tb[5][70] = torch.tensor([0.2, 0.7, 0.2001, 0.7001])
    tb[6][10] = tb[6][1000].clone()
    d = sumG - B * 1024
    if d < 0:
        tb[0], tc[0] = tb[0][:1024 + d].contiguous(), tc[0][:1024 + d].contiguous()
    elif d > 0:                                                 # late duplicates of early gts
        tb[0], tc[0] = torch.cat([tb[0], tb[0][:d]]), torch.cat([tc[0], tc[0][:d]])
    assert sum(int(b.shape[0]) for b in tb) == sumG
    return tb, tc


@pytest.mark.parametrize("sumG", [OBJ_MAP_MAX, SEED_CAP, SEED_CAP + 1])
def test_gts_per_batch_across_the_16_bit_switches(sumG):
    from objectdetection_ssd_b200 import _lib
    from objectdetection_ssd_b200.head import PackedGT
    pri = H.priors()
    P = pri.shape[0]
    B = 64
    tb, tc = _dense_gt_batch(sumG)
    loc, conf = synth.make_head(302, B, P)
    loc, conf = torch.from_numpy(loc), torch.from_numpy(conf)
    _check_match(_head(pri), pri, tb, tc)                              # standalone match kernel
    torch.cuda.synchronize()
    n0 = _launches()
    out, ref = _check_loss(pri, loc, conf, tb, tc)                     # two-kernel step
    launches = _launches() - n0
    obj_map, cull = sumG <= OBJ_MAP_MAX, sumG <= SEED_CAP
    # the step: [seed kernel of the cull] + streaming kernel + mining kernel with the fused finaliser (cooperative)
    assert launches == 2 + int(cull), f"{launches} launches: not the two-kernel step with the cull {'on' if cull else 'off'}"
    assert torch.equal(out["cls_u8"].cpu().long(), ref["cls"])
    assert torch.equal(out["best_prior"][:sumG].cpu().long(), ref["best_prior"])
    # most priors are positive: 3 x npos exceeds the negatives, every negative is mined
    mined = H.unpack_mask(out["mined_mask"], P)
    assert bool((3 * ref["npos"] >= (~ref["pos"]).sum(1)).all())
    assert torch.equal(mined, ~ref["pos"]), "mining did not take every negative"
    print(f"[limits] sumG = {sumG}: best-gt map {'on' if obj_map else 'off (finaliser walks the gts)'}, "
          f"seeded cull {'on' if cull else 'off'}, {launches} launches, npos {int(ref['npos'].min())}..{int(ref['npos'].max())} "
          f"of {P}, mining saturated")
    if sumG <= SEED_CAP:
        return
    # three-kernel route (what a batch that does not fit co-resident uses): ce_match_stream + finaliser + mining kernel
    head = _head(pri)
    gt = PackedGT(tb, tc, head.dev)
    lib = head.lib
    m = head._match_outputs(gt, False)
    ws = head._workspace(_lib.WS_LOSS, B, 0)
    wm = head._workspace(_lib.WS_MATCH, B, gt.sumG)
    st = torch.cuda.current_stream().cuda_stream
    l, c = loc.cuda(), conf.cuda()
    gl, gcf = torch.empty_like(l), torch.empty_like(c)
    sums = torch.empty(2, dtype=torch.float64, device="cuda")
    losses = torch.empty(2, device="cuda")
    _lib.check(lib.ssdhead_ce_match_stream(c.data_ptr(), gt.boxes.data_ptr(), gt.classes.data_ptr(), gt.off.data_ptr(),
                                           head.pri_xyxy.data_ptr(), B, P, 21, gt.sumG, 0.5, None, gl.data_ptr(), gcf.data_ptr(),
                                           m["cls_u8"].data_ptr(), m["best_prior"].data_ptr(), m["npos"].data_ptr(),
                                           ws.data_ptr(), ws.numel(), wm.data_ptr(), wm.numel(), 1, st), "ce_match_stream")
    _lib.check(lib.ssdhead_mine(l.data_ptr(), c.data_ptr(), gt.boxes.data_ptr(), gt.classes.data_ptr(), gt.off.data_ptr(),
                                head.pri_xyxy.data_ptr(), head.pri_cxcywh.data_ptr(), m["best_prior"].data_ptr(),
                                m["npos"].data_ptr(), m["npos"][B:].data_ptr(), m["cls_u8"].data_ptr(), B, P, 21, 3, 0.5,
                                sums.data_ptr(), losses.data_ptr(), gl.data_ptr(), gcf.data_ptr(), None, None,
                                ws.data_ptr(), ws.numel(), st), "mine")
    torch.cuda.synchronize()
    assert torch.equal(m["cls_u8"], out["cls_u8"]) and torch.equal(m["npos"], out["npos"])
    assert torch.equal(m["best_prior"][:sumG], out["best_prior"][:sumG])
    assert torch.equal(gcf, out["grad_conf"]) and torch.equal(gl, out["grad_loc"])
    assert torch.equal(losses, out["losses"])
    print(f"[limits] sumG = {sumG}: three-kernel route gives the same bits")


# ---------------------------------------------------------------------------------------------------------------------
# 3. detect at the largest prior count

DET_P_MAX = 512 * 256    # score tiles of 256 rows, at most one per thread of the 512-thread sweep CTA
DET_BIAS, DET_MIN = 6.0, 0.03     # ~60 000 candidates per ordinary image at this prior count (~3 000 per class)


@pytest.mark.parametrize("P", [DET_P_MAX, DET_P_MAX - 1])
def test_detect_at_the_largest_prior_count(P):
    from objectdetection_ssd_b200.head import detect, detect_fallbacks, detect_from_scores
    pri = _prior_table(DET_P_MAX, seed=1)[:P].contiguous()
    head = _head(pri)
    loc, conf = H.detect_inputs(401, 2, P, bg_bias=DET_BIAS)
    boxes = torch.stack([O.decode(loc[i], pri) for i in range(2)])
    probs = F.softmax(conf, dim=2)
    # one clustered image: two classes of ~4 400 heavily overlapping candidates each -> the sweep runs through many slices
    cb, cp = _clustered_inputs(402, 1, pri, classes=(2, 11), frac=4400 / P)
    boxes, probs = torch.cat([boxes, cb]).contiguous(), torch.cat([probs, cp]).contiguous()
    B = 3
    ncand = [int((probs[i, :, :20] >= DET_MIN).sum()) for i in range(B)]
    assert all(10_000 <= n <= 100_000 for n in ncand[:2]) and ncand[2] > 8000, ncand
    ref = _oracle_stage(boxes, probs, DET_MIN, 0.45, 200)
    outs, nfb = {}, {}
    for shortlist in (False, True):
        with _route(shortlist):
            outs[shortlist] = detect_from_scores(head, boxes, probs, DET_MIN, 0.45, 200)
            nfb[shortlist] = detect_fallbacks(head, B)
        torch.cuda.synchronize()
        _check_exact(outs[shortlist], ref, 200)
    _same(outs[True], outs[False])
    assert nfb[False] == 0
    cnt = outs[True]["cnt"].cpu().tolist()
    print(f"[limits] detect at P = {P}: candidates per image {ncand}, detections {cnt}, "
          f"short-list fallbacks {nfb[True]} of {B}; both routes equal the oracle")
    # fused path (own softmax + decode) on the ordinary images, both routes
    fused = {}
    for shortlist in (False, True):
        with _route(shortlist):
            fused[shortlist] = detect(head, loc, conf, DET_MIN, 0.45, 200)
            nf = detect_fallbacks(head, 2)
        torch.cuda.synchronize()
        if shortlist:
            print(f"[limits] fused detect at P = {P}: short-list fallbacks {nf} of 2")
    _same(fused[True], fused[False])
    n = H.compare_detect_with_oracle(fused[True], loc, conf, pri, DET_MIN, 0.45, 200, range(2))
    print(f"[limits] fused detect at P = {P}: {n} detections differ from the oracle, all with a boundary proof")


def test_detect_one_prior_past_the_limit_is_refused_before_any_launch():
    from objectdetection_ssd_b200.head import detect, detect_from_scores
    P = DET_P_MAX + 1
    pri = _prior_table(P, seed=1)
    head = _head(pri)
    loc, conf = H.detect_inputs(403, 1, P, bg_bias=DET_BIAS)
    l, c = loc.cuda(), conf.cuda()
    torch.cuda.synchronize()
    n0 = _launches()
    for fn in (detect, detect_from_scores):
        for shortlist in (False, True):
            with _route(shortlist), pytest.raises(RuntimeError, match=r"unsupported shape.*code -2"):
                fn(head, l, c, DET_MIN, 0.45, 200)
    assert _launches() == n0, "a refused call launched kernels"
    print(f"[limits] detect at P = {P}: refused (E_UNSUPPORTED), no launch")


# ---------------------------------------------------------------------------------------------------------------------
# 4. detect at the largest accepted top_k

def _detect_accepts(head, boxes, probs, top_k):
    from objectdetection_ssd_b200.head import detect_from_scores
    try:
        detect_from_scores(head, boxes, probs, 0.5, 0.45, top_k)
    except RuntimeError as e:
        assert "code -2" in str(e), e
        return False
    return True


@pytest.fixture(scope="module")
def top_k_max():
    """Largest top_k an SSD300 call accepts, bisected with calls on one image without candidates (the shape checks
    refuse before any launch)."""
    pri = H.priors()
    head = _head(pri)
    boxes = pri.unsqueeze(0).contiguous()
    probs = torch.zeros(1, pri.shape[0], 21)
    probs[..., 20] = 1.0
    lo, hi = 600, 60001
    assert _detect_accepts(head, boxes, probs, lo) and not _detect_accepts(head, boxes, probs, hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if _detect_accepts(head, boxes, probs, mid) else (lo, mid)
    torch.cuda.synchronize()
    print(f"\n[limits] detect (SSD300 priors): top_k_max = {lo}")
    return lo


def test_detect_at_the_largest_top_k(top_k_max):
    from objectdetection_ssd_b200.head import detect, detect_fallbacks, detect_from_scores
    K = top_k_max
    pri = H.priors()
    P = pri.shape[0]
    head = _head(pri)
    B = 3
    loc, conf = H.detect_inputs(501, B, P, bg_bias=6.0)
    boxes = torch.stack([O.decode(loc[i], pri) for i in range(B)])
    probs = F.softmax(conf, dim=2)
    ncand = [int((probs[i, :, :20] >= 0.01).sum()) for i in range(B)]
    ref = _oracle_stage(boxes, probs, 0.01, 0.45, K)
    with _route(True):
        fast = detect_from_scores(head, boxes, probs, 0.01, 0.45, K)
        nfb = detect_fallbacks(head, B)
    with _route(False):
        full = detect_from_scores(head, boxes, probs, 0.01, 0.45, K)
        nfb0 = detect_fallbacks(head, B)
    torch.cuda.synchronize()
    _same(fast, full)
    _check_exact(fast, ref, K)
    cnt = fast["cnt"].cpu().tolist()
    print(f"[limits] detect at top_k = {K}: candidates per image {ncand}, detections {cnt}, "
          f"short-list fallbacks {nfb} of {B}")
    assert (fast["cnt"].cpu() == K).all()               # more than top_k survive: the global cut is exercised
    # The short list is sized from a sample of every 35th row (about 1 600 keys expected, SAMPLE_TARGET in csrc/detect.cu):
    # at this top_k an image is decided by it only when its sampled floor happens to list more than top_k + 1
    # survivors, so most images need the fallback (2 of these 3); either way the output above is the oracle's.
    assert nfb >= 1, "no image took the fallback: the short list of an image cannot decide this top_k"
    assert nfb0 == 0
    # the fused path on both routes
    with _route(True):
        a = detect(head, loc, conf, 0.01, 0.45, K)
        assert detect_fallbacks(head, B) >= 1
    with _route(False):
        b = detect(head, loc, conf, 0.01, 0.45, K)
    torch.cuda.synchronize()
    _same(a, b)
    # one more is refused before any launch, on both routes
    n0 = _launches()
    for shortlist in (False, True):
        with _route(shortlist), pytest.raises(RuntimeError, match=r"unsupported shape.*code -2"):
            detect_from_scores(head, boxes, probs, 0.01, 0.45, K + 1)
    assert _launches() == n0, "a refused call launched kernels"


# ---------------------------------------------------------------------------------------------------------------------
# 5. get_map at evaluation scale

def _eval_set(n_img=400, seed=601):
    """Detections of ``Losses.inference_batch`` (top_k 200) on SSD300 head outputs that partly find the gts, plus
    adversarial images and edits.  Returns (det boxes, det classes, det scores, gt boxes, gt classes) as lists."""
    from objectdetection_ssd_b200 import Losses
    pri = H.priors()
    P = pri.shape[0]
    gb, gc = synth.make_gt(seed, n_img, 1, 8)
    tb, tc = [torch.from_numpy(b) for b in gb], [torch.from_numpy(c) for c in gc]
    loc, conf = synth.make_head(seed + 1, n_img, P)
    loc, conf = torch.from_numpy(loc), torch.from_numpy(conf)
    m = O.match_batch(tb, tc, O.cxcywh_to_xyxy(pri))
    g = torch.Generator().manual_seed(seed + 2)
    conf = conf * 0.1
    conf[..., 20] += 4.0
    gt_cxcywh = O.xyxy_to_cxcywh(torch.cat(tb))
    for b in range(n_img):
        p = m["pos"][b].nonzero().flatten()
        conf[b, p, m["cls"][b, p]] += 2.0 + 7.0 * torch.rand(p.numel(), generator=g)
        # noisy box regressions: some detections land below IoU 0.5 with their gt
        loc[b, p] = O.encode(gt_cxcywh[m["obj"][b, p]], pri[p]) + 0.6 * torch.randn(p.numel(), 4, generator=g)
    out = Losses.inference_batch(loc.cuda(), conf.cuda(), top_k=200, min_score=0.01)
    torch.cuda.synchronize()
    cnt = out["cnt"].cpu()
    db = [out["boxes"][b, :int(cnt[b])].cpu() for b in range(n_img)]
    dc = [out["cls"][b, :int(cnt[b])].cpu().long() for b in range(n_img)]
    # scores quantised to multiples of 1/64: ties inside and across images (rank ties -> lower detection index)
    ds = [torch.round(out["prob"][b, :int(cnt[b])].cpu() * 64) / 64 for b in range(n_img)]
    # class 19 has gts and no detection at all
    for b in range(n_img):
        keep = dc[b] != 19
        db[b], dc[b], ds[b] = db[b][keep], dc[b][keep], ds[b][keep]
    # an image with detections of classes it has no gt of
    db.append(torch.tensor([[0.1, 0.1, 0.4, 0.4], [0.5, 0.5, 0.9, 0.9], [0.1, 0.1, 0.4, 0.4]]))
    dc.append(torch.tensor([3, 7, 0]))
    ds.append(torch.tensor([1.0, 0.75, 0.5]))
    tb.append(torch.tensor([[0.6, 0.1, 0.9, 0.3]]))
    tc.append(torch.tensor([0.]))
    # an image without gts, with detections
    db.append(torch.tensor([[0.2, 0.2, 0.5, 0.5], [0.3, 0.3, 0.6, 0.6]]))
    dc.append(torch.tensor([5, 8]))
    ds.append(torch.tensor([0.984375, 0.984375]))
    tb.append(torch.zeros(0, 4))
    tc.append(torch.zeros(0))
    # several detections claiming one gt (only the first in rank order is a true positive)
    gbox = torch.tensor([0.3, 0.2, 0.7, 0.6])
    db.append(torch.stack([gbox, gbox + 0.01, gbox - 0.01, gbox, gbox + torch.tensor([0.02, 0.0, 0.02, 0.0])]))
    dc.append(torch.full((5,), 8))
    ds.append(torch.tensor([0.5, 1.0, 0.75, 1.0, 0.25]))
    tb.append(gbox.unsqueeze(0))
    tc.append(torch.tensor([8.]))
    # a detection whose IoU with its gt is exactly 0.5 (every quantity dyadic): not a true positive (IoU > 0.5 is)
    g5 = torch.tensor([[0.25, 0.25, 0.75, 0.75]])
    d5 = torch.tensor([[0.25, 0.25, 0.75, 0.5]])
    assert float(O.iou_matrix(d5, g5)[0, 0]) == 0.5
    db.append(d5)
    dc.append(torch.tensor([5]))
    ds.append(torch.tensor([0.999]))
    tb.append(g5)
    tc.append(torch.tensor([5.]))
    return db, dc, ds, tb, tc


def test_get_map_at_evaluation_scale():
    from objectdetection_ssd_b200 import Util
    db, dc, ds, tb, tc = _eval_set()
    N = sum(int(d.shape[0]) for d in db)
    M = sum(int(t.shape[0]) for t in tb)
    assert N > 65536, N
    gt_classes = set(int(x) for t in tc for x in t.tolist())
    assert gt_classes == set(range(20))
    det_per_class = np.bincount(torch.cat(dc).numpy(), minlength=20)
    assert det_per_class[19] == 0 and (det_per_class[:19] > 0).all()
    got = Util.get_map(db, dc, ds, tb, tc)
    want = O.voc_ap(db, dc, ds, tb, tc)
    got = np.array([got[c] for c in range(20)])
    print(f"[limits] get_map: {len(db)} images, {N} detections, {M} gts; AP {np.round(got, 4).tolist()}")
    assert np.array_equal(got, want), (got, want)
    assert want[19] == 0.0
    assert 0.05 < want[:19].mean() < 0.95                 # neither trivial nor perfect
