"""CUDA graph capture of the training-head step and detect.

``sumG`` is a capacity: with gt arrays longer than the batch (a tail of NaN boxes and class 255) every entry point
gives the bits of the exact call.  ``StaticHead`` captured around loss + backward, loss_levels, detect or a whole SGD
step replays what the eager drop-in calls compute, bit for bit, with new gts loaded before each replay.  The host-list
calls and ``PackedGT`` refuse a capture.
"""
import os
import subprocess
import sys

import pytest
import torch

from objectdetection_ssd_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SENTINEL = -7


def _lists(seed, B, lo, hi):
    gb, gc = synth.make_gt(seed, B, lo, hi)
    return [torch.from_numpy(b) for b in gb], [torch.from_numpy(c) for c in gc]


def _head_in(seed, B, P):
    loc, conf = synth.make_head(seed, B, P)
    return torch.from_numpy(loc).cuda(), torch.from_numpy(conf).cuda()


def _priors():
    from objectdetection_ssd_b200 import Losses
    return Losses.ancs_xywh


def _capacity_gt(gt, cap):
    """The gts of a PackedGT in buffers of `cap` rows, the tail filled with NaN boxes and class 255."""
    from objectdetection_ssd_b200.head import _StaticGT
    s = _StaticGT(gt.B, cap, gt.boxes.device)
    s.boxes.fill_(float("nan"))
    s.classes.fill_(255.0)
    s.boxes[:gt.sumG].copy_(gt.boxes)
    s.classes[:gt.sumG].copy_(gt.classes)
    s.off.copy_(gt.off)
    return s


def _step(head, l, c, gt):
    """ssdhead_multibox_step with every output and tap, best_prior pre-filled with a sentinel."""
    from objectdetection_ssd_b200 import _lib
    B, P, lib = l.shape[0], head.P, head.lib
    ws = torch.zeros(int(lib.ssdhead_workspace_bytes(_lib.WS_LOSS, B, P, 21, 0)), dtype=torch.uint8, device="cuda")
    wm = torch.zeros(int(lib.ssdhead_workspace_bytes(_lib.WS_MATCH, B, P, 21, gt.sumG)), dtype=torch.uint8, device="cuda")
    o = dict(sums=torch.empty(2, dtype=torch.float64, device="cuda"), losses=torch.empty(2, device="cuda"),
             grad_loc=torch.empty_like(l), grad_conf=torch.empty_like(c),
             cls_u8=torch.empty(B, P, dtype=torch.uint8, device="cuda"),
             best_prior=torch.full((gt.sumG,), SENTINEL, dtype=torch.int32, device="cuda"),
             npos=torch.empty(B + 1, dtype=torch.int32, device="cuda"),
             mined=torch.empty(B, (P + 31) // 32, dtype=torch.int32, device="cuda"),
             ce=torch.empty(B, P, device="cuda"))
    _lib.check(lib.ssdhead_multibox_step(
        l.data_ptr(), c.data_ptr(), gt.boxes.data_ptr(), gt.classes.data_ptr(), gt.off.data_ptr(),
        head.pri_xyxy.data_ptr(), head.pri_cxcywh.data_ptr(), B, P, 21, gt.sumG, 3, 0.5,
        o["sums"].data_ptr(), o["losses"].data_ptr(), o["grad_loc"].data_ptr(), o["grad_conf"].data_ptr(),
        o["cls_u8"].data_ptr(), o["best_prior"].data_ptr(), o["npos"].data_ptr(), o["mined"].data_ptr(),
        o["ce"].data_ptr(), ws.data_ptr(), ws.numel(), wm.data_ptr(), wm.numel(), torch.cuda.current_stream().cuda_stream),
        "ssdhead_multibox_step")
    torch.cuda.synchronize()
    assert int(wm.count_nonzero()) == 0, "the match workspace was not left zeroed"
    return o


def _same(a, b, n, what):
    for k in a:
        x, y = a[k], b[k]
        if k == "best_prior":
            assert torch.equal(x[:n], y[:n]), f"{what}: best_prior"
            continue
        assert torch.equal(x, y), f"{what}: {k}"


# ---------------------------------------------------------------------------------------------------------------------
# 1. sumG is a capacity

@pytest.mark.parametrize("case", ["ordinary", "cull", "map_off", "B300"])
def test_capacity_gives_the_bits_of_the_exact_count(case, monkeypatch):
    from objectdetection_ssd_b200.head import MultiboxHead, PackedGT
    head = MultiboxHead(_priors(), "cuda")
    B, lo, hi, extra = {"ordinary": (16, 1, 10, 777), "cull": (16, 20, 40, 333), "map_off": (32, 1, 10, 70000),
                        "B300": (300, 1, 10, 1000)}[case]
    if case == "cull":
        monkeypatch.setenv("SSDHEAD_MATCH_CULL_MIN", "1")
    tb, tc = _lists(11, B, lo, hi)
    l, c = _head_in(11, B, head.P)
    gt = PackedGT(tb, tc, head.dev)
    n = gt.sumG
    cap = _capacity_gt(gt, n + extra)
    if case == "map_off":
        assert n <= 65535 < cap.sumG
    exact = _step(head, l, c, gt)
    got = _step(head, l, c, cap)
    _same(exact, got, n, case)
    assert bool((got["best_prior"][n:] == SENTINEL).all()), "best_prior written past gt_off[B]"
    assert int(exact["npos"][-1]) > 0


@pytest.mark.parametrize("cull", ["24", "1"])
def test_capacity_levels_resident_and_match(cull, monkeypatch):
    from objectdetection_ssd_b200.ctx import SSDHeadContext
    from objectdetection_ssd_b200.head import MultiboxHead, PackedGT
    monkeypatch.setenv("SSDHEAD_MATCH_CULL_MIN", cull)
    head = MultiboxHead(_priors(), "cuda")
    B, P = 12, head.P
    tb, tc = _lists(12, B, 1, 30)
    l, c = _head_in(12, B, P)
    gt = PackedGT(tb, tc, head.dev)
    n = gt.sumG
    cap = _capacity_gt(gt, n + 500)
    # levels step
    counts, s0, ll, cl = (5776, 2166, 600, 150, 36, 4), 0, [], []
    for k in counts:
        ll.append(l[:, s0:s0 + k].contiguous())
        cl.append(c[:, s0:s0 + k].contiguous())
        s0 += k
    a = head.loss_levels(ll, cl, gt, with_grads=True)
    b = head.loss_levels(ll, cl, cap, with_grads=True)
    torch.cuda.synchronize()
    for k in ("losses", "sums", "npos", "cls_u8"):
        assert torch.equal(a[k], b[k]), f"levels: {k}"
    assert torch.equal(a["best_prior"][:n], b["best_prior"][:n])
    for x, y in zip(a["grad_loc"] + a["grad_conf"], b["grad_loc"] + b["grad_conf"]):
        assert torch.equal(x, y), "levels: gradients"
    # ssdhead_match
    outs = head._match_outputs(cap, True)
    outs["best_prior"].fill_(SENTINEL)
    mc = head.match(cap, want_maps=True, outs=outs)
    me = head.match(gt, want_maps=True)
    torch.cuda.synchronize()
    for k in ("npos", "cls_u8", "obj", "cls"):
        assert torch.equal(me[k], mc[k]), f"match: {k}"
    assert torch.equal(me["best_prior"], mc["best_prior"][:n])
    assert bool((mc["best_prior"][n:] == SENTINEL).all())
    # resident step (through the context: sumG = capacity) against the dense step with the exact count
    ctx = SSDHeadContext(_priors().numpy(), max_batch=B, max_total_gt=cap.sumG)
    st = torch.cuda.current_stream().cuda_stream
    gl_r, gc_r = torch.empty_like(l), torch.empty_like(c)
    sr, lr = torch.empty(2, dtype=torch.float64, device="cuda"), torch.empty(2, device="cuda")
    gl_d, gc_d = torch.empty_like(l), torch.empty_like(c)
    sd, ld = torch.empty(2, dtype=torch.float64, device="cuda"), torch.empty(2, device="cuda")
    ctx.loss_dev_resident(l.data_ptr(), c.data_ptr(), cap.boxes.data_ptr(), cap.classes.data_ptr(), cap.off.data_ptr(), B,
                          cap.sumG, sr.data_ptr(), lr.data_ptr(), gl_r.data_ptr(), gc_r.data_ptr(), st, fresh=True)
    ctx.loss_dev(l.data_ptr(), c.data_ptr(), gt.boxes.data_ptr(), gt.classes.data_ptr(), gt.off.data_ptr(), B, n,
                 sd.data_ptr(), ld.data_ptr(), gl_d.data_ptr(), gc_d.data_ptr(), st)
    torch.cuda.synchronize()
    assert torch.equal(lr, ld) and torch.equal(sr, sd)
    assert torch.equal(gl_r, gl_d) and torch.equal(gc_r, gc_d)
    assert torch.equal(ld, a["losses"])
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2.-3., 7. StaticHead replays against the eager drop-in calls

PLAN = [(1, 1), (5, 15), (32, 32), (1, 1), (5, 15), (32, 32)]       # gts per image (lo, hi); 32 per image = max_gt


def _warm_and_capture(fn):
    """One eager call on a side stream (allocates the workspaces), then the capture; returns (graph, outputs)."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fn()
    return g, out


def _workspaces_clean(sh):
    from objectdetection_ssd_b200 import _lib
    torch.cuda.synchronize()
    wm = sh.head._ws[_lib.WS_MATCH]
    wl = sh.head._ws[_lib.WS_LOSS]
    assert int(wm.count_nonzero()) == 0, "match workspace not zero after the replays"
    assert int(wl[:16].count_nonzero()) == 0, "loss workspace counter not zero after the replays"


@pytest.mark.parametrize("B", [32, 256])
def test_captured_loss_and_backward_replay_eager_ssd(B):
    from objectdetection_ssd_b200 import Losses
    from objectdetection_ssd_b200.Losses import StaticHead
    P = _priors().shape[0]
    sh = StaticHead(_priors(), B, 32 * B, "cuda")
    l0, c0 = _head_in(100, B, P)
    loc, conf = l0.clone().requires_grad_(), c0.clone().requires_grad_()
    tb, tc = _lists(100, B, 3, 8)
    sh.load(tb, tc)

    def step():
        loc.grad = conf.grad = None
        a, b = sh.loss(loc, conf)
        (a + b).backward()
        return a, b

    g, (la, lb) = _warm_and_capture(step)
    for i, (lo, hi) in enumerate(PLAN):
        tb, tc = _lists(200 + i, B, lo, hi)
        if lo == 32:
            assert sum(t.shape[0] for t in tb) == sh.max_gt
        if i % 2:
            sh.load([t.cuda() for t in tb], [t.cuda() for t in tc])        # device lists
        else:
            sh.load(tb, tc)
        nl, nc = _head_in(200 + i, B, P)
        with torch.no_grad():
            loc.copy_(nl)
            conf.copy_(nc)
        g.replay()
        el, ec = nl.clone().requires_grad_(), nc.clone().requires_grad_()
        ea, eb = Losses.ssd((el, ec), tc, tb)
        (ea + eb).backward()
        torch.cuda.synchronize()
        assert torch.equal(la, ea) and torch.equal(lb, eb), f"replay {i}: losses"
        assert torch.equal(loc.grad, el.grad) and torch.equal(conf.grad, ec.grad), f"replay {i}: gradients"
    _workspaces_clean(sh)


@pytest.mark.parametrize("B", [32, 256])
def test_captured_loss_levels_replay_eager_ssd_levels(B):
    from objectdetection_ssd_b200 import Losses
    from objectdetection_ssd_b200.Losses import StaticHead
    from objectdetection_ssd_b200.collate import collate_gt
    P = _priors().shape[0]
    counts = (5776, 2166, 600, 150, 36, 4)
    sh = StaticHead(_priors(), B, 32 * B, "cuda")

    def split(l, c):
        s0, ll, cl = 0, [], []
        for k in counts:
            ll.append(l[:, s0:s0 + k].contiguous())
            cl.append(c[:, s0:s0 + k].contiguous())
            s0 += k
        return ll, cl

    locs, confs = split(*_head_in(300, B, P))
    for t in locs + confs:
        t.requires_grad_()
    sh.load_packed(*collate_gt(*_lists(300, B, 1, 9)))

    def step():
        for t in locs + confs:
            t.grad = None
        a, b = sh.loss_levels(locs, confs)
        (a + b).backward()
        return a, b

    g, (la, lb) = _warm_and_capture(step)
    for i, (lo, hi) in enumerate(PLAN):
        tb, tc = _lists(400 + i, B, lo, hi)
        sh.load_packed(*collate_gt(tb, tc))
        nl, nc = split(*_head_in(400 + i, B, P))
        with torch.no_grad():
            for d, s in zip(locs + confs, nl + nc):
                d.copy_(s)
        g.replay()
        el = [t.clone().requires_grad_() for t in nl]
        ec = [t.clone().requires_grad_() for t in nc]
        ea, eb = Losses.ssd_levels((el, ec), tc, tb)
        (ea + eb).backward()
        torch.cuda.synchronize()
        assert torch.equal(la, ea) and torch.equal(lb, eb), f"replay {i}: losses"
        for x, y in zip(locs + confs, el + ec):
            assert torch.equal(x.grad, y.grad), f"replay {i}: gradients"
    _workspaces_clean(sh)


@pytest.mark.parametrize("B", [8, 256])
def test_captured_detect_replays_eager_inference_batch(B):
    from objectdetection_ssd_b200 import Losses
    from objectdetection_ssd_b200.Losses import StaticHead
    P = _priors().shape[0]
    sh = StaticHead(_priors(), B, B, "cuda")
    loc, conf = (t.clone() for t in _head_in(500, B, P))
    wh = torch.tensor([[300.0 + i, 200.0 + 2 * i] for i in range(B)], device="cuda")
    for use_wh in (False, True):
        g, out = _warm_and_capture(lambda: sh.detect(loc, conf, 0.01, 0.45, 200, img_wh=wh if use_wh else None))
        for i in range(3):
            l, c = synth.make_head(600 + i, B, P, loc_scale=0.5, bg_bias=4.0 + i)
            loc.copy_(torch.from_numpy(l))
            conf.copy_(torch.from_numpy(c))
            g.replay()
            ref = Losses.inference_batch(loc.clone(), conf.clone(), top_k=200, min_score=0.01, iou_threshold=0.45,
                                         img_wh=wh if use_wh else None)
            torch.cuda.synchronize()
            assert torch.equal(out["cnt"], ref["cnt"]), f"replay {i}: counts"
            assert int(ref["cnt"].sum()) > 0
            for b in range(B):
                k = int(ref["cnt"][b])
                for key in ("boxes", "prob", "cls", "prior"):
                    assert torch.equal(out[key][b, :k], ref[key][b, :k]), f"replay {i}, image {b}: {key}"
        del g


# ---------------------------------------------------------------------------------------------------------------------
# 4. a whole training step

def test_captured_training_step_equals_eager_steps():
    from objectdetection_ssd_b200 import Losses
    from objectdetection_ssd_b200.Losses import StaticHead
    B, P, lr = 16, _priors().shape[0], 0.5
    fl, fc = _head_in(700, B, P)                               # fixed features of a per-channel affine "model"

    def params():
        return [torch.ones(4, device="cuda", requires_grad=True), torch.zeros(4, device="cuda", requires_grad=True),
                torch.ones(21, device="cuda", requires_grad=True), torch.zeros(21, device="cuda", requires_grad=True)]

    def forward(p, xl, xc):
        return xl * p[0] + p[1], xc * p[2] + p[3]

    def sgd(p):
        with torch.no_grad():
            for t in p:
                t.sub_(lr * t.grad)

    batches = [_lists(710 + i, B, 1, 12) for i in range(5)]
    feats = [_head_in(720 + i, B, P) for i in range(5)]

    pe = params()                                             # eager
    for (tb, tc), (xl, xc) in zip(batches, feats):
        for t in pe:
            t.grad = None
        a, b = Losses.ssd(forward(pe, xl, xc), tc, tb)
        (a + b).backward()
        sgd(pe)

    pg = params()                                             # captured
    sh = StaticHead(_priors(), B, 12 * B, "cuda")
    sh.load(*_lists(709, B, 1, 12))
    init = [t.detach().clone() for t in pg]

    def step():
        for t in pg:
            t.grad = None
        a, b = sh.loss(*forward(pg, fl, fc))
        (a + b).backward()
        sgd(pg)

    g, _ = _warm_and_capture(step)
    with torch.no_grad():                                     # undo the warm-up step
        for t, v in zip(pg, init):
            t.copy_(v)
    for (tb, tc), (xl, xc) in zip(batches, feats):
        sh.load(tb, tc)
        fl.copy_(xl)
        fc.copy_(xc)
        g.replay()
    torch.cuda.synchronize()
    for x, y in zip(pg, pe):
        assert torch.equal(x, y), "parameters after five replays differ from five eager steps"
    assert not torch.equal(pe[2], torch.ones(21, device="cuda"))


# ---------------------------------------------------------------------------------------------------------------------
# 5. the first mining launch of a process inside a capture

CHILD = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
from objectdetection_ssd_b200 import Losses, _lib, synth
from objectdetection_ssd_b200.Losses import StaticHead
B = 64
pri = Losses.ancs_xywh
P = pri.shape[0]
sh = StaticHead(pri, B, 40 * B, "cuda")
sh.head._workspace(_lib.WS_LOSS, B, 0)                  # workspaces allocated eagerly, no kernel launched
sh.head._workspace(_lib.WS_MATCH, B, sh.max_gt)
def lists(seed, lo, hi):
    gb, gc = synth.make_gt(seed, B, lo, hi)
    return [torch.from_numpy(b) for b in gb], [torch.from_numpy(c) for c in gc]
def head_in(seed):
    l, c = synth.make_head(seed, B, P)
    return torch.from_numpy(l).cuda(), torch.from_numpy(c).cuda()
l0, c0 = head_in(1)
loc, conf = l0.clone().requires_grad_(), c0.clone().requires_grad_()
sh.load(*lists(1, 1, 10))
torch.cuda.synchronize()
n0 = _lib.launch_count()
g = torch.cuda.CUDAGraph()
with torch.cuda.graph(g):
    a, b = sh.loss(loc, conf)
    (a + b).backward()
assert _lib.launch_count() > n0
for i, (lo, hi) in enumerate([(1, 10), (30, 40), (1, 1)]):
    tb, tc = lists(10 + i, lo, hi)
    sh.load(tb, tc)
    nl, nc = head_in(10 + i)
    with torch.no_grad():
        loc.copy_(nl); conf.copy_(nc)
    g.replay()
    el, ec = nl.clone().requires_grad_(), nc.clone().requires_grad_()
    ea, eb = Losses.ssd((el, ec), tc, tb)
    (ea + eb).backward()
    torch.cuda.synchronize()
    assert torch.equal(a, ea) and torch.equal(b, eb), i
    assert torch.equal(loc.grad, el.grad) and torch.equal(conf.grad, ec.grad), i
print("ok")
"""


def test_first_mining_launch_of_a_process_inside_a_capture():
    res = subprocess.run([sys.executable, "-c", CHILD, ROOT], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert res.returncode == 0 and res.stdout.strip().endswith("ok"), res.stdout + res.stderr


# ---------------------------------------------------------------------------------------------------------------------
# 6. C callers: the context's device entry points with sumG = max_sumG

def test_captured_context_steps_replay_eager_steps():
    from objectdetection_ssd_b200.ctx import SSDHeadContext
    from objectdetection_ssd_b200.head import _StaticGT, PackedGT
    B, P = 48, _priors().shape[0]
    cap = 40 * B
    pri = _priors().numpy()
    ctx = SSDHeadContext(pri, max_batch=B, max_total_gt=cap)         # captured
    ref = SSDHeadContext(pri, max_batch=B, max_total_gt=cap)         # eager, exact counts
    gt = _StaticGT(B, cap, torch.device("cuda", torch.cuda.current_device()))
    loc, conf = (t.clone() for t in _head_in(800, B, P))
    f32 = lambda *s: torch.empty(*s, device="cuda")
    sums, losses, gl, gc = torch.empty(2, dtype=torch.float64, device="cuda"), f32(2), f32(B, P, 4), f32(B, P, 21)
    sums_r, losses_r = torch.empty(2, dtype=torch.float64, device="cuda"), f32(2)
    gl_r, gc_r = torch.zeros(B, P, 4, device="cuda"), torch.zeros(B, P, 21, device="cuda")

    def load(tb, tc):
        p = PackedGT(tb, tc, gt.block.device)
        gt.boxes[:p.sumG].copy_(p.boxes)
        gt.classes[:p.sumG].copy_(p.classes)
        gt.off.copy_(p.off)
        return p

    load(*_lists(800, B, 1, 10))

    def step(fresh=False):
        st = torch.cuda.current_stream().cuda_stream
        ctx.loss_dev(loc.data_ptr(), conf.data_ptr(), gt.boxes.data_ptr(), gt.classes.data_ptr(), gt.off.data_ptr(), B, cap,
                     sums.data_ptr(), losses.data_ptr(), gl.data_ptr(), gc.data_ptr(), st)
        ctx.loss_dev_resident(loc.data_ptr(), conf.data_ptr(), gt.boxes.data_ptr(), gt.classes.data_ptr(), gt.off.data_ptr(),
                              B, cap, sums_r.data_ptr(), losses_r.data_ptr(), gl_r.data_ptr(), gc_r.data_ptr(), st, fresh=fresh)

    step(fresh=True)                                          # eager: hands the resident tensors over
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step()
    st = torch.cuda.current_stream().cuda_stream
    for i, (lo, hi) in enumerate([(1, 1), (5, 15), (40, 40), (1, 3)]):
        p = load(*_lists(810 + i, B, lo, hi))
        nl, nc = _head_in(810 + i, B, P)
        loc.copy_(nl)
        conf.copy_(nc)
        g.replay()
        s_e, l_e, gl_e, gc_e = torch.empty(2, dtype=torch.float64, device="cuda"), f32(2), f32(B, P, 4), f32(B, P, 21)
        ref.loss_dev(nl.data_ptr(), nc.data_ptr(), p.boxes.data_ptr(), p.classes.data_ptr(), p.off.data_ptr(), B, p.sumG,
                     s_e.data_ptr(), l_e.data_ptr(), gl_e.data_ptr(), gc_e.data_ptr(), st)
        torch.cuda.synchronize()
        assert torch.equal(losses, l_e) and torch.equal(sums, s_e), f"replay {i}: loss_dev losses"
        assert torch.equal(gl, gl_e) and torch.equal(gc, gc_e), f"replay {i}: loss_dev gradients"
        assert torch.equal(losses_r, l_e) and torch.equal(sums_r, s_e), f"replay {i}: resident losses"
        assert torch.equal(gl_r, gl_e) and torch.equal(gc_r, gc_e), f"replay {i}: resident gradients"
    ctx.close()
    ref.close()


# ---------------------------------------------------------------------------------------------------------------------
# 8. refusals

@pytest.mark.filterwarnings("ignore:The CUDA Graph is empty")
def test_host_list_calls_refuse_a_capture():
    from objectdetection_ssd_b200 import Losses
    from objectdetection_ssd_b200.head import PackedGT
    B, P = 2, _priors().shape[0]
    tb, tc = _lists(900, B, 1, 3)
    l, c = _head_in(900, B, P)
    wh = (300, 200)
    lv = [l[:, :5776], l[:, 5776:]], [c[:, :5776], c[:, 5776:]]
    calls = {
        "ssd": lambda: Losses.ssd((l, c), tc, tb),
        "ssd_levels": lambda: Losses.ssd_levels(lv, tc, tb),
        "ssd1_": lambda: Losses.ssd1_(l, c, tb, tc),
        "ssd1": lambda: Losses.ssd1(l[0], c[0], tb[0], tc[0]),
        "ssd_old": lambda: Losses.ssd_old((l, c), tc, tb),
        "inference": lambda: Losses.inference(l[0], c[0], wh, toDraw=False),
        "inference_batch": lambda: Losses.inference_batch(l, c),
        "inference_batch_levels": lambda: Losses.inference_batch_levels(*lv),
        "PackedGT": lambda: PackedGT(tb, tc, l.device),
    }
    torch.cuda.synchronize()
    for name, fn in calls.items():
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            with pytest.raises(RuntimeError, match="StaticHead"):
                fn()
        del g
    # eager: unchanged
    a, b = Losses.ssd((l, c), tc, tb)
    assert torch.isfinite(a) and torch.isfinite(b)


@pytest.mark.filterwarnings("ignore:The CUDA Graph is empty")
def test_static_head_refusals():
    from objectdetection_ssd_b200.Losses import StaticHead
    B, P = 4, _priors().shape[0]
    sh = StaticHead(_priors(), B, 20, "cuda")
    tb, tc = _lists(950, B, 5, 5)
    with pytest.raises(RuntimeError, match="load"):
        sh.loss(*_head_in(950, B, P))                         # nothing loaded yet
    sh.load(tb, tc)                                           # exactly max_gt
    with pytest.raises(ValueError, match="max_gt"):
        sh.load(*_lists(951, B, 6, 6))
    with pytest.raises(ValueError, match="4 images"):
        sh.load(tb[:3], tc[:3])
    with pytest.raises(IndexError, match="image 2"):
        sh.load(tb[:2] + [torch.zeros(0, 4)] + tb[3:], tc[:2] + [torch.zeros(0)] + tc[3:])
    from objectdetection_ssd_b200.collate import collate_gt
    gx, gcl, off = collate_gt(tb, tc)
    bad = off.copy()
    bad[2] = bad[1]
    with pytest.raises(IndexError, match="image 1"):
        sh.load_packed(gx, gcl, bad)
    l, c = _head_in(950, B, P)
    with pytest.raises(ValueError, match="img_wh"):
        sh.detect(l, c, img_wh=torch.ones(B, 2))
    g = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        with pytest.raises(RuntimeError, match="outside the graph"):
            sh.load(tb, tc)
        with pytest.raises(RuntimeError, match="outside the graph"):
            sh.load_packed(gx, gcl, off)
        with pytest.raises(RuntimeError, match="warm-up"):
            sh.loss(l, c)                                     # first call: allocates its workspace
        with pytest.raises(RuntimeError, match="warm-up"):
            sh.detect(l, c)
    del g
    a, b = sh.loss(l, c)                                      # eager after the refusals: works
    torch.cuda.synchronize()
    assert torch.isfinite(a) and torch.isfinite(b)
