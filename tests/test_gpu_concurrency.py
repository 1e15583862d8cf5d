"""GPU: the head path under concurrency.  The device entry points keep no global state and are re-entrant across streams
when each call has its own workspace (include/ssdhead.h); a MultiboxHead orders its own workspaces between streams and
threads; every front end runs on the device of its tensors.  Each case enqueues everything first, synchronises once and
compares every concurrent result bit for bit with the same call run serially (with a synchronise after each), over
rounds of changing inputs; one case per group is also held against the oracle, so that "equal to the serial run" cannot
mean "equally wrong".  After the rounds one more serial call per workspace still gives the serial bits: the
self-resetting counters were left zeroed."""
import ctypes
import os
import threading

import numpy as np
import pytest
import torch

from objectdetection_ssd_b200 import _lib, synth
from oracle import ssd_oracle as O
from tests import helpers as H

pytestmark = pytest.mark.gpu

C = 21
ROUNDS = 3
LEVEL_COUNTS = (5776, 2166, 600, 150, 36, 4)          # SSD300's six levels (sum 8732)


def _dev(a, dev="cuda"):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _zeros_ws(lib, which, B, P, n, dev="cuda"):
    return torch.zeros(int(lib.ssdhead_workspace_bytes(which, B, P, C, n)) + 256, dtype=torch.uint8, device=dev)


def _p(t):
    return None if t is None else t.data_ptr()


def _assert_same(got: dict, want: dict, what: str):
    assert got.keys() == want.keys(), what
    for k in want:
        a, b = got[k], want[k]
        if isinstance(b, torch.Tensor):
            assert a.dtype == b.dtype and a.shape == b.shape, f"{what}: {k} {a.dtype}{tuple(a.shape)} vs {b.dtype}{tuple(b.shape)}"
            same = torch.equal(a.cpu(), b.cpu()) or bool(torch.equal(torch.isnan(a.cpu()), torch.isnan(b.cpu())) and
                                                         torch.equal(torch.nan_to_num(a.cpu()), torch.nan_to_num(b.cpu())))
            assert same, f"{what}: {k} differs from the serial run"
        else:
            assert a == b, f"{what}: {k} {a} vs {b}"


class _Gate:
    """Holds streams back while the host enqueues a round, so that their work really overlaps once released (the host
    is slower to enqueue a call than the GPU is to run it): they wait on an event recorded behind ordinary copies of a
    few GB on a third stream - several milliseconds of memory traffic."""

    def __init__(self, gb=2, copies=12):
        self.src = torch.empty(gb << 30, dtype=torch.uint8, device="cuda")
        self.dst = torch.empty_like(self.src)
        self.copies = copies
        self.stream = torch.cuda.Stream()

    def hold(self, *streams):
        with torch.cuda.stream(self.stream):
            for _ in range(self.copies):
                self.dst.copy_(self.src)
        ev = torch.cuda.Event()
        ev.record(self.stream)
        for st in streams:
            st.wait_event(ev)


def _serial(fn, *args):
    """fn(*args) on the current stream, complete when it returns."""
    out = fn(*args)
    torch.cuda.synchronize()
    return out


# ------------------------------------------------------------------------------------------------ inputs of a round
class _Round:
    """Head outputs and gts of up to 300 SSD300 images, and detect inputs of 256, on the device; seeded."""

    def __init__(self, seed, pri, dev="cuda"):
        P = pri.shape[0]
        self.P, self.dev = P, dev
        self.gb, self.gc = synth.make_gt(seed, 300)
        loc, conf = synth.make_head(seed, 300, P)
        self.loc, self.conf = _dev(loc, dev), _dev(conf, dev)
        dl, dc = synth.make_head(seed + 1000, 256, P, loc_scale=0.5, bg_bias=6.0)
        self.dloc, self.dconf = _dev(dl, dev), _dev(dc, dev)
        self._gt = {}
        self._levels = {}

    def gt(self, B):
        if B not in self._gt:
            gx, gcl, off = synth.pack_gt(self.gb[:B], self.gc[:B])
            self._gt[B] = (_dev(gx, self.dev), _dev(gcl, self.dev), _dev(off, self.dev), int(off[-1]))
        return self._gt[B]

    def levels(self, B):
        """Per-level dense copies of the first B images' loc / conf."""
        if B not in self._levels:
            locs, confs, a = [], [], 0
            for n in LEVEL_COUNTS:
                locs.append(self.loc[:B, a:a + n].contiguous())
                confs.append(self.conf[:B, a:a + n].contiguous())
                a += n
            self._levels[B] = (locs, confs)
        return self._levels[B]


class _Priors:
    def __init__(self, pri, dev="cuda"):
        self.cxcywh = pri.to(dev).contiguous()
        self.xyxy = O.cxcywh_to_xyxy(pri).to(dev).contiguous()
        self.P = int(pri.shape[0])


# ------------------------------------------------------------------------------------------------ A: raw ABI jobs
# Each job owns its workspaces (zero-filled once, reused every round) and returns fresh output tensors per call.
class _Step:
    """ssdhead_multibox_step (B <= co-resident capacity: two kernels; B = 300: the three-kernel route)."""

    def __init__(self, lib, pr, B):
        self.lib, self.pr, self.B = lib, pr, B
        self.ws = _zeros_ws(lib, _lib.WS_LOSS, B, pr.P, 0)
        self.wm = _zeros_ws(lib, _lib.WS_MATCH, B, pr.P, 10 * B)

    def __call__(self, r, st):
        B, P, pr = self.B, self.pr.P, self.pr
        gx, gcl, off, n = r.gt(B)
        o = dict(sums=torch.empty(2, dtype=torch.float64, device="cuda"), losses=torch.empty(2, device="cuda"),
                 gl=torch.empty(B, P, 4, device="cuda"), gc=torch.empty(B, P, C, device="cuda"),
                 cls=torch.empty(B, P, dtype=torch.uint8, device="cuda"),
                 bp=torch.empty(max(n, 1), dtype=torch.int32, device="cuda"),
                 npos=torch.empty(B + 1, dtype=torch.int32, device="cuda"))
        _lib.check(self.lib.ssdhead_multibox_step(
            _p(r.loc), _p(r.conf), _p(gx), _p(gcl), _p(off), _p(pr.xyxy), _p(pr.cxcywh), B, P, C, n, 3, 0.5,
            _p(o["sums"]), _p(o["losses"]), _p(o["gl"]), _p(o["gc"]), _p(o["cls"]), _p(o["bp"]), _p(o["npos"]),
            None, None, _p(self.ws), self.ws.numel(), _p(self.wm), self.wm.numel(), st.cuda_stream),
            f"ssdhead_multibox_step B={B}")
        return o


class _Resident:
    """ssdhead_multibox_step_resident: the gradient tensors persist between calls; each call's copy is taken in stream
    order."""

    def __init__(self, lib, pr, B):
        self.lib, self.pr, self.B = lib, pr, B
        self.ws = _zeros_ws(lib, _lib.WS_LOSS, B, pr.P, 0)
        self.wm = _zeros_ws(lib, _lib.WS_MATCH, B, pr.P, 10 * B)
        self.rows = _zeros_ws(lib, _lib.WS_ROWS, B, pr.P, 0)
        self.gl = torch.zeros(B, pr.P, 4, device="cuda")
        self.gc = torch.zeros(B, pr.P, C, device="cuda")

    def __call__(self, r, st):
        B, P, pr = self.B, self.pr.P, self.pr
        gx, gcl, off, n = r.gt(B)
        o = dict(sums=torch.empty(2, dtype=torch.float64, device="cuda"), losses=torch.empty(2, device="cuda"),
                 cls=torch.empty(B, P, dtype=torch.uint8, device="cuda"),
                 bp=torch.empty(max(n, 1), dtype=torch.int32, device="cuda"),
                 npos=torch.empty(B + 1, dtype=torch.int32, device="cuda"))
        _lib.check(self.lib.ssdhead_multibox_step_resident(
            _p(r.loc), _p(r.conf), _p(gx), _p(gcl), _p(off), _p(pr.xyxy), _p(pr.cxcywh), B, P, C, n, 3, 0.5,
            _p(o["sums"]), _p(o["losses"]), _p(self.gl), _p(self.gc), _p(o["cls"]), _p(o["bp"]), _p(o["npos"]),
            _p(self.ws), self.ws.numel(), _p(self.wm), self.wm.numel(), _p(self.rows), self.rows.numel(),
            1, 0, 0, None, None, None, st.cuda_stream), "ssdhead_multibox_step_resident")
        with torch.cuda.stream(st):
            o["gl"], o["gc"] = self.gl.clone(), self.gc.clone()
        return o


class _Levels:
    """ssdhead_multibox_step_levels on SSD300's six level tensors."""

    def __init__(self, lib, pr, B):
        self.lib, self.pr, self.B = lib, pr, B
        self.ws = _zeros_ws(lib, _lib.WS_LOSS, B, pr.P, 0)
        self.wm = _zeros_ws(lib, _lib.WS_MATCH, B, pr.P, 10 * B)

    def __call__(self, r, st):
        B, P, pr = self.B, self.pr.P, self.pr
        gx, gcl, off, n = r.gt(B)
        locs, confs = r.levels(B)
        gls = [torch.empty_like(t) for t in locs]
        gcs = [torch.empty_like(t) for t in confs]
        lv = _lib.Levels()
        lv.num_levels = len(LEVEL_COUNTS)
        for i, cnt in enumerate(LEVEL_COUNTS):
            lv.count[i], lv.conf[i], lv.loc[i] = cnt, confs[i].data_ptr(), locs[i].data_ptr()
            lv.grad_conf[i], lv.grad_loc[i] = gcs[i].data_ptr(), gls[i].data_ptr()
        o = dict(sums=torch.empty(2, dtype=torch.float64, device="cuda"), losses=torch.empty(2, device="cuda"),
                 cls=torch.empty(B, P, dtype=torch.uint8, device="cuda"),
                 bp=torch.empty(max(n, 1), dtype=torch.int32, device="cuda"),
                 npos=torch.empty(B + 1, dtype=torch.int32, device="cuda"))
        _lib.check(self.lib.ssdhead_multibox_step_levels(
            ctypes.addressof(lv), _p(gx), _p(gcl), _p(off), _p(pr.xyxy), _p(pr.cxcywh), B, P, C, n, 3, 0.5,
            _p(o["sums"]), _p(o["losses"]), _p(o["cls"]), _p(o["bp"]), _p(o["npos"]),
            _p(self.ws), self.ws.numel(), _p(self.wm), self.wm.numel(), st.cuda_stream), "ssdhead_multibox_step_levels")
        o["gl"], o["gc"] = gls, gcs
        return o


class _StreamMineSparse:
    """ssdhead_ce_match_stream (no gradient pointers) then ssdhead_mine_sparse: packed gradient rows."""

    ROW_CAP = 2048

    def __init__(self, lib, pr, B):
        self.lib, self.pr, self.B = lib, pr, B
        self.ws = _zeros_ws(lib, _lib.WS_LOSS, B, pr.P, 0)
        self.wm = _zeros_ws(lib, _lib.WS_MATCH, B, pr.P, 10 * B)

    def __call__(self, r, st):
        B, P, pr, cap = self.B, self.pr.P, self.pr, self.ROW_CAP
        gx, gcl, off, n = r.gt(B)
        o = dict(sums=torch.empty(2, dtype=torch.float64, device="cuda"), losses=torch.empty(2, device="cuda"),
                 cls=torch.empty(B, P, dtype=torch.uint8, device="cuda"),
                 bp=torch.empty(max(n, 1), dtype=torch.int32, device="cuda"),
                 npos=torch.empty(B + 1, dtype=torch.int32, device="cuda"),
                 cnt=torch.empty(B, 2, dtype=torch.int32, device="cuda"),
                 idx=torch.full((B, cap), -1, dtype=torch.int32, device="cuda"),
                 rc=torch.zeros(B, cap, C, device="cuda"), rl=torch.zeros(B, cap, 4, device="cuda"))
        _lib.check(self.lib.ssdhead_ce_match_stream(
            _p(r.conf), _p(gx), _p(gcl), _p(off), _p(pr.xyxy), B, P, C, n, 0.5, None, None, None,
            _p(o["cls"]), _p(o["bp"]), _p(o["npos"]), _p(self.ws), self.ws.numel(), _p(self.wm), self.wm.numel(), 1,
            st.cuda_stream), "ssdhead_ce_match_stream")
        _lib.check(self.lib.ssdhead_mine_sparse(
            _p(r.loc), _p(r.conf), _p(gx), _p(gcl), _p(off), _p(pr.xyxy), _p(pr.cxcywh),
            _p(o["bp"]), _p(o["npos"]), o["npos"].data_ptr() + 4 * B, _p(o["cls"]), B, P, C, 3, 0.5,
            _p(o["sums"]), _p(o["losses"]), cap, _p(o["cnt"]), _p(o["idx"]), _p(o["rc"]), _p(o["rl"]),
            _p(self.ws), self.ws.numel(), st.cuda_stream), "ssdhead_mine_sparse")
        return o

    @staticmethod
    def canonical(o):
        """The row order inside an image is unspecified (the set is not): rows sorted by prior index, positives first."""
        o = {k: v.cpu() for k, v in o.items()}
        cnt, idx, rc, rl = o.pop("cnt"), o.pop("idx"), o.pop("rc"), o.pop("rl")
        assert int(cnt[:, 0].max()) <= _StreamMineSparse.ROW_CAP
        for b in range(cnt.shape[0]):
            n, npos = int(cnt[b, 0]), int(cnt[b, 1])
            for part, (a, z) in (("pos", (0, npos)), ("neg", (npos, n))):
                order = torch.argsort(idx[b, a:z].long()) + a
                o[f"{b}{part}_idx"] = idx[b, order]
                o[f"{b}{part}_conf"] = rc[b, order]
                if part == "pos":
                    o[f"{b}{part}_loc"] = rl[b, order]
        o["cnt"] = cnt
        return o


class _Detect:
    """ssdhead_detect at B = 256 on one route (the route switch is read per call)."""

    def __init__(self, lib, pr, B, shortlist, top_k=200):
        self.lib, self.pr, self.B, self.route, self.top_k = lib, pr, B, "1" if shortlist else "0", top_k
        self.ws = _zeros_ws(lib, _lib.WS_DETECT, B, pr.P, 0)

    def __call__(self, r, st):
        B, K = self.B, self.top_k
        o = dict(boxes=torch.empty(B, K, 4, device="cuda"), prob=torch.empty(B, K, device="cuda"),
                 cls=torch.empty(B, K, dtype=torch.int32, device="cuda"),
                 prior=torch.empty(B, K, dtype=torch.int32, device="cuda"),
                 cnt=torch.empty(B, dtype=torch.int32, device="cuda"))
        old = os.environ.get("SSDHEAD_DETECT_SHORTLIST")
        os.environ["SSDHEAD_DETECT_SHORTLIST"] = self.route
        try:
            _lib.check(self.lib.ssdhead_detect(
                _p(r.dloc[:B]), _p(r.dconf[:B]), _p(self.pr.cxcywh), B, self.pr.P, C, 0.01, 0.45, K, None, 0,
                _p(o["boxes"]), _p(o["prob"]), _p(o["cls"]), _p(o["prior"]), _p(o["cnt"]),
                _p(self.ws), self.ws.numel(), st.cuda_stream), f"ssdhead_detect route {self.route}")
        finally:
            if old is None:
                os.environ.pop("SSDHEAD_DETECT_SHORTLIST", None)
            else:
                os.environ["SSDHEAD_DETECT_SHORTLIST"] = old
        return o


def _voc_inputs(seed, n_img=24):
    g = np.random.default_rng(seed)
    det_b, det_c, det_s, gt_b, gt_c = [], [], [], [], []
    for _ in range(n_img):
        m = int(g.integers(1, 6))
        xy = g.uniform(0, 0.7, (m, 2)).astype(np.float32)
        gb = np.concatenate([xy, xy + g.uniform(0.05, 0.3, (m, 2)).astype(np.float32)], 1)
        gc = g.integers(0, 20, m).astype(np.float32)
        k = int(g.integers(0, 12))
        src = g.integers(0, m, k)
        db = gb[src] + g.normal(0, 0.03, (k, 4)).astype(np.float32)
        dc = np.where(g.random(k) < 0.8, gc[src], g.integers(0, 20, k)).astype(np.int64)
        ds = np.round(g.random(k), 2).astype(np.float32)                 # ties on purpose
        det_b.append(torch.from_numpy(db)); det_c.append(torch.from_numpy(dc)); det_s.append(torch.from_numpy(ds))
        gt_b.append(torch.from_numpy(gb)); gt_c.append(torch.from_numpy(gc))
    return det_b, det_c, det_s, gt_b, gt_c


class _VocAp:
    def __init__(self, lib):
        self.lib = lib
        self.levels = torch.arange(0, 1.1, 0.1).to(device="cuda", dtype=torch.float64)

    def prepare(self, seed):
        db, dc, ds, gb, gc = _voc_inputs(seed)
        doff = np.concatenate([[0], np.cumsum([len(x) for x in db])]).astype(np.int32)
        goff = np.concatenate([[0], np.cumsum([len(x) for x in gb])]).astype(np.int32)
        self.raw = (db, dc, ds, gb, gc)
        self.t = (torch.cat(db).cuda(), torch.cat(dc).to("cuda", torch.int32), torch.cat(ds).cuda(), _dev(doff), int(doff[-1]),
                  torch.cat(gb).cuda(), torch.cat(gc).cuda(), _dev(goff), int(goff[-1]), len(db))
        N, M = self.t[4], self.t[8]
        self.ws = torch.empty(int(self.lib.ssdhead_voc_ap_workspace_bytes(N, M, 20)), dtype=torch.uint8, device="cuda")

    def __call__(self, r, st):
        db, dc, ds, doff, N, gb, gc, goff, M, n = self.t
        ap = torch.full((20,), -1.0, dtype=torch.float64, device="cuda")
        _lib.check(self.lib.ssdhead_voc_ap(_p(db), _p(dc), _p(ds), _p(doff), N, _p(gb), _p(gc), _p(goff), M, n, 20, 0.5,
                                           _p(self.levels), _p(ap), _p(self.ws), self.ws.numel(), st.cuda_stream),
                   "ssdhead_voc_ap")
        return dict(ap=ap)


def _detections(o):
    """A detect output without its padding (what lies past cnt[b] is not written)."""
    if "cnt" not in o:
        return o
    o = dict(o)
    cnt = o["cnt"]
    keep = torch.arange(o["prob"].shape[1], device=cnt.device)[None, :] < cnt.clamp(min=0)[:, None]
    for k in ("boxes", "prob", "cls", "prior"):
        if k in o:
            o[k] = o[k][keep]
    return o


def _canon(name, o):
    if name == "mine_sparse":
        return _StreamMineSparse.canonical(o)
    o = _detections(o)
    out = {}
    for k, v in o.items():
        if isinstance(v, list):
            for i, t in enumerate(v):
                out[f"{k}{i}"] = t.cpu()
        else:
            out[k] = v.cpu()
    return out


def test_raw_abi_two_streams_separate_workspaces():
    """A: every device entry point, two streams (one of high priority), each call with its own workspace: the
    concurrent results are the serial ones; the B = 64 step and the short-list detect agree with the oracle."""
    lib = _lib.load()
    pri = H.priors()
    pr = _Priors(pri)

    def jobs():
        return {"step256": _Step(lib, pr, 256), "step64": _Step(lib, pr, 64), "step300": _Step(lib, pr, 300),
                "resident": _Resident(lib, pr, 64), "levels": _Levels(lib, pr, 64),
                "mine_sparse": _StreamMineSparse(lib, pr, 64),
                "detect_short": _Detect(lib, pr, 256, True), "detect_full": _Detect(lib, pr, 256, False),
                "voc": _VocAp(lib)}
    # the streams of the concurrent run: a training step always has a detect or another step beside it
    lanes = {"hi": ["step256", "detect_full", "resident", "step300", "voc"],
             "lo": ["detect_short", "step64", "levels", "mine_sparse"]}
    serial, conc = jobs(), jobs()
    torch.cuda.synchronize()
    s_hi = torch.cuda.Stream(priority=-1)
    s_lo = torch.cuda.Stream()
    cur = torch.cuda.current_stream()
    gate = _Gate()
    first = None
    for rnd in range(ROUNDS):
        r = _Round(100 + rnd, pri)
        for j in (serial, conc):
            j["voc"].prepare(200 + rnd)
        torch.cuda.synchronize()
        want = {k: _canon(k, _serial(serial[k], r, cur)) for k in serial}
        got = {}
        gate.hold(s_hi, s_lo)
        for i in range(max(len(v) for v in lanes.values())):       # interleave the two lanes' enqueues
            for lane, st in (("hi", s_hi), ("lo", s_lo)):
                if i < len(lanes[lane]):
                    k = lanes[lane][i]
                    with torch.cuda.stream(st):
                        got[k] = conc[k](r, st)
        torch.cuda.synchronize()
        for k in want:
            _assert_same(_canon(k, got[k]), want[k], f"round {rnd}: {k}")
        if rnd == 0:
            first = (r, want)
            # the oracle: the B = 64 step's losses, and the short-list route's detections of a few images
            tb = [torch.from_numpy(b) for b in r.gb[:64]]
            tc = [torch.from_numpy(c) for c in r.gc[:64]]
            ref = O.multibox_loss(r.loc[:64].cpu(), r.conf[:64].cpu(), tb, tc, pri)
            losses = want["step64"]["losses"]
            assert abs(losses[0].item() - ref["loc_loss"].item()) <= 1e-5 * abs(ref["loc_loss"].item())
            assert abs(losses[1].item() - ref["conf_loss"].item()) <= 1e-5 * abs(ref["conf_loss"].item())
            assert int(want["step64"]["npos"][-1]) == ref["npos_total"]
            out = {k: v for k, v in got["detect_short"].items()}
            H.compare_detect_with_oracle(out, r.dloc.cpu(), r.dconf.cpu(), pri, 0.01, 0.45, 200, range(3))
            ap = O.voc_ap(*conc["voc"].raw)
            assert np.array_equal(got["voc"]["ap"].cpu().numpy(), np.asarray(ap, dtype=np.float64))
    # one more serial call per workspace, on the first round's inputs
    r, want = first
    for j in (serial, conc):
        j["voc"].prepare(200)
    torch.cuda.synchronize()
    for k in conc:
        _assert_same(_canon(k, _serial(conc[k], r, cur)), want[k], f"serial call after the rounds: {k}")


# ------------------------------------------------------------------------------------------------ B: one head, two streams
def _head_outputs(out):
    keep = ("losses", "sums", "npos", "grad_loc", "grad_conf", "best_prior", "cls_u8", "boxes", "prob", "cls", "prior",
            "cnt")
    res = {}
    for k, v in _detections(out).items():
        if k in keep and v is not None:
            res[k] = torch.cat(v, 1) if isinstance(v, list) else v
    return res


def _head_calls(head, r, Losses):
    """The calls of case B, in order: (name, fn) - each returns a dict of tensors."""
    from objectdetection_ssd_b200.head import PackedGT, detect
    tb = lambda B: [torch.from_numpy(b) for b in r.gb[:B]]
    tc = lambda B: [torch.from_numpy(c) for c in r.gc[:B]]

    def loss(B):
        return lambda: _head_outputs(head.loss(r.loc[:B], r.conf[:B], PackedGT(tb(B), tc(B), head.dev), with_grads=True))

    def levels(B):
        def f():
            locs, confs = r.levels(B)
            return _head_outputs(head.loss_levels(locs, confs, PackedGT(tb(B), tc(B), head.dev), with_grads=True))
        return f

    def det(B, k):
        return lambda: _head_outputs(detect(head, r.dloc[:B], r.dconf[:B], 0.01, 0.45, k))

    def ssd(B):
        def f():
            l1, l2 = Losses.ssd((r.loc[:B], r.conf[:B]), tc(B), tb(B))
            return dict(loc_loss=l1.detach().clone(), conf_loss=l2.detach().clone())
        return f

    def inf(B):
        return lambda: _head_outputs(Losses.inference_batch(r.dloc[:B], r.dconf[:B], 200, 0.01, 0.45))

    # batch sizes change from call to call on purpose: every change re-zeroes a workspace, some grow it
    return [("loss64", loss(64)), ("levels32", levels(32)), ("detect256", det(256, 200)), ("loss128", loss(128)),
            ("detect64", det(64, 200)), ("levels64", levels(64)), ("ssd32", ssd(32)), ("infer128", inf(128)),
            ("ssd256", ssd(256)), ("infer64", inf(64)), ("loss32", loss(32))]


def test_one_head_two_streams_without_synchronize():
    """B: one MultiboxHead (and the drop-in surface's head) used from two streams with no synchronise between the
    calls: the head orders its workspaces between the streams, so every result is the serial one."""
    from objectdetection_ssd_b200 import Losses
    from objectdetection_ssd_b200.head import MultiboxHead
    pri = H.priors()
    s1, s2 = torch.cuda.Stream(priority=-1), torch.cuda.Stream()
    gate = _Gate()
    head_serial, head = MultiboxHead(pri, "cuda"), MultiboxHead(pri, "cuda")
    saved = Losses.ancs_xywh
    Losses.ancs_xywh = pri
    try:
        first = None
        for rnd in range(ROUNDS):
            r = _Round(300 + rnd, pri)
            r.levels(32), r.levels(64)
            torch.cuda.synchronize()
            Losses._heads.clear()
            want = {name: _serial(fn) for name, fn in _head_calls(head_serial, r, Losses)}
            Losses._heads.clear()
            got = {}
            gate.hold(s1, s2)
            for i, (name, fn) in enumerate(_head_calls(head, r, Losses)):
                with torch.cuda.stream(s1 if i % 2 == 0 else s2):
                    got[name] = fn()
            torch.cuda.synchronize()
            for name in want:
                _assert_same(got[name], want[name], f"round {rnd}: {name}")
            if rnd == 0:
                first = (r, want)
                tb = [torch.from_numpy(b) for b in r.gb[:32]]
                tc = [torch.from_numpy(c) for c in r.gc[:32]]
                ref = O.multibox_loss(r.loc[:32].cpu(), r.conf[:32].cpu(), tb, tc, pri)
                lo = want["loss32"]["losses"].cpu()
                assert abs(lo[0].item() - ref["loc_loss"].item()) <= 1e-5 * abs(ref["loc_loss"].item())
                assert abs(lo[1].item() - ref["conf_loss"].item()) <= 1e-5 * abs(ref["conf_loss"].item())
        r, want = first
        for name, fn in _head_calls(head, r, Losses):
            _assert_same(_serial(fn), want[name], f"serial call after the rounds: {name}")
    finally:
        Losses.ancs_xywh = saved
        Losses._heads.clear()


# ------------------------------------------------------------------------------------------------ C: host threads
def _run_threads(targets):
    errors = []

    def wrap(fn):
        def run():
            try:
                torch.cuda.set_device(0)
                fn()
            except BaseException as e:          # noqa: BLE001 - re-raised in the main thread
                errors.append(e)
        return run
    ts = [threading.Thread(target=wrap(fn)) for fn in targets]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    if errors:
        raise errors[0]


class _ThreadWork:
    """One thread's model: its own head and stream, a loss step and a detect per step on a few input sets."""

    def __init__(self, kind, B, top_k, seed, nsets=3):
        from objectdetection_ssd_b200.head import MultiboxHead
        self.pri = H.priors(kind)
        self.P, self.B, self.top_k = self.pri.shape[0], B, top_k
        self.head = MultiboxHead(self.pri, "cuda")
        self.sets = []
        for i in range(nsets):
            gb, gc = synth.make_gt(seed + i, B, 1, 10 if kind == "ssd300" else 100)
            loc, conf = synth.make_head(seed + i, B, self.P)
            dl, dc = synth.make_head(seed + 50 + i, B, self.P, loc_scale=0.5, bg_bias=6.0)
            self.sets.append(([torch.from_numpy(b) for b in gb], [torch.from_numpy(c) for c in gc],
                              _dev(loc), _dev(conf), _dev(dl), _dev(dc)))

    def step(self, i):
        from objectdetection_ssd_b200.head import PackedGT, detect
        tb, tc, loc, conf, dl, dc = self.sets[i % len(self.sets)]
        out = _head_outputs(self.head.loss(loc, conf, PackedGT(tb, tc, self.head.dev), with_grads=True))
        out.update({f"det_{k}": v for k, v in _head_outputs(detect(self.head, dl, dc, 0.01, 0.45, self.top_k)).items()})
        return out


def test_two_threads_two_models_with_their_own_heads():
    """C: two host threads, each with its own head and stream - SSD300 (P = 8732) with detect at top_k 200 beside
    SSD512 (P = 24564, 100 gts per image) with top_k 1000, 100 steps each: the kernels' launch settings are per device
    and fixed, so neither thread's shapes disturb the other's launches; every step gives the serial bits."""
    steps = 100
    works = [_ThreadWork("ssd300", 16, 200, 400), _ThreadWork("ssd512", 8, 1000, 500)]
    want = [[_serial(w.step, i) for i in range(len(w.sets))] for w in works]
    got = [[None] * steps for _ in works]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    torch.cuda.synchronize()

    def runner(t):
        def run():
            with torch.cuda.stream(streams[t]):
                for i in range(steps):
                    got[t][i] = works[t].step(i)
        return run
    _run_threads([runner(0), runner(1)])
    torch.cuda.synchronize()
    for t, w in enumerate(works):
        for i in range(steps):
            _assert_same(got[t][i], want[t][i % len(w.sets)], f"thread {t} step {i}")
    # the oracle on the SSD512 thread's first set (its detect at top_k 1000 on a few images; the serial bits above)
    from objectdetection_ssd_b200.head import detect
    w = works[1]
    _, _, _, _, dl, dc = w.sets[0]
    out = _serial(detect, w.head, dl, dc, 0.01, 0.45, 1000)
    assert all(torch.equal(v.cpu(), want[1][0][f"det_{k}"].cpu()) for k, v in _detections(out).items())
    H.compare_detect_with_oracle(out, dl.cpu(), dc.cpu(), w.pri, 0.01, 0.45, 1000, range(2))
    for t, w in enumerate(works):
        _assert_same(_serial(w.step, 0), want[t][0], f"thread {t}: serial call after the threads")


def test_two_threads_two_host_contexts():
    """C: two SSDHeadContexts (SSD300 and SSD512) running loss_host / detect_host from two threads."""
    from objectdetection_ssd_b200.ctx import SSDHeadContext, pinned_empty
    cfgs = [("ssd300", 8, 200, 600), ("ssd512", 4, 1000, 700)]
    models = []
    for kind, B, k, seed in cfgs:
        pri = H.priors(kind)
        P = pri.shape[0]
        sets = []
        for i in range(2):
            gb, gc = synth.make_gt(seed + i, B)
            loc, conf = synth.make_head(seed + i, B, P, loc_scale=0.5, bg_bias=6.0)
            hl, hc = pinned_empty(loc.shape), pinned_empty(conf.shape)
            hl[:], hc[:] = loc, conf
            sets.append((hl, hc) + synth.pack_gt(gb, gc))
        models.append((SSDHeadContext(pri.numpy(), max_batch=B, top_k=k), sets, B, P, k))

    def call(m, i):
        ctx, sets, B, P, k = m
        hl, hc, gx, gcl, off = sets[i % len(sets)]
        gl, gcf = np.empty((B, P, 4), np.float32), np.empty((B, P, C), np.float32)
        l1, l2 = ctx.loss_host(hl, hc, gx, gcl, off, gl, gcf)
        ob, op = pinned_empty((B, k, 4)), pinned_empty((B, k))
        oc, oi, on = pinned_empty((B, k), np.int32), pinned_empty((B, k), np.int32), pinned_empty((B,), np.int32)
        ctx.detect_host(hl, hc, ob, op, oc, oi, on, 0.01, 0.45)
        det = [(ob[b, :on[b]].copy(), op[b, :on[b]].copy(), oc[b, :on[b]].copy(), oi[b, :on[b]].copy())
               for b in range(B)]
        return (l1, l2), gl, gcf, on.copy(), det

    def same(a, b, what):
        assert a[0] == b[0], what
        assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2]), what
        assert np.array_equal(a[3], b[3]), what
        for x, y in zip(a[4], b[4]):
            assert all(np.array_equal(u, v) for u, v in zip(x, y)), what

    want = [[call(m, i) for i in range(2)] for m in models]
    # the SSD300 context against the oracle (losses)
    ctx, sets, B, P, _ = models[0]
    hl, hc, gx, gcl, off = sets[0]
    gb, gc = synth.make_gt(600, B)
    ref = O.multibox_loss(torch.from_numpy(np.array(hl)), torch.from_numpy(np.array(hc)),
                          [torch.from_numpy(b) for b in gb], [torch.from_numpy(c) for c in gc], H.priors())
    assert abs(want[0][0][0][0] - ref["loc_loss"].item()) <= 1e-5 * abs(ref["loc_loss"].item())
    assert abs(want[0][0][0][1] - ref["conf_loss"].item()) <= 1e-5 * abs(ref["conf_loss"].item())
    n = 12
    got = [[None] * n for _ in models]

    def runner(t):
        def run():
            for i in range(n):
                got[t][i] = call(models[t], i)
        return run
    _run_threads([runner(0), runner(1)])
    for t in range(len(models)):
        for i in range(n):
            same(got[t][i], want[t][i % 2], f"context {t} call {i}")
    for m in models:
        m[0].close()


def test_two_threads_drop_in_ssd_with_host_gt_lists():
    """C: two threads calling Losses.ssd with host gt lists (the pinned staging pool) on their own streams, one shared
    drop-in head: every call gives its serial losses and gradients."""
    from objectdetection_ssd_b200 import Losses
    pri = H.priors()
    saved = Losses.ancs_xywh
    Losses.ancs_xywh = pri
    try:
        sets = []
        for i in range(4):
            B = (16, 24, 16, 32)[i]
            gb, gc = synth.make_gt(800 + i, B)
            loc, conf = synth.make_head(800 + i, B, pri.shape[0])
            sets.append(([torch.from_numpy(c) for c in gc], [torch.from_numpy(b) for b in gb], _dev(loc), _dev(conf)))

        def call(i):
            tc, tb, loc, conf = sets[i % len(sets)]
            l = loc.clone().requires_grad_(True)
            c = conf.clone().requires_grad_(True)
            l1, l2 = Losses.ssd((l, c), tc, tb)
            (l1 + l2).backward()
            return dict(l1=l1.detach(), l2=l2.detach(), gl=l.grad, gc=c.grad)

        want = [_serial(call, i) for i in range(len(sets))]
        ref = O.multibox_loss(sets[0][2].cpu(), sets[0][3].cpu(), sets[0][1], sets[0][0], pri)
        assert abs(want[0]["l1"].item() - ref["loc_loss"].item()) <= 1e-5 * abs(ref["loc_loss"].item())
        assert abs(want[0]["l2"].item() - ref["conf_loss"].item()) <= 1e-5 * abs(ref["conf_loss"].item())
        n = 24
        got = [[None] * n for _ in range(2)]
        streams = [torch.cuda.Stream(), torch.cuda.Stream()]
        torch.cuda.synchronize()

        def runner(t):
            def run():
                with torch.cuda.stream(streams[t]):
                    for i in range(n):
                        got[t][i] = call(i + t)
            return run
        _run_threads([runner(0), runner(1)])
        torch.cuda.synchronize()
        for t in range(2):
            for i in range(n):
                _assert_same(got[t][i], want[(i + t) % len(sets)], f"thread {t} call {i}")
    finally:
        Losses.ancs_xywh = saved
        Losses._heads.clear()


# ------------------------------------------------------------------------------------------------ D: a second device
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_second_device_while_device_0_is_current():
    """D: the front ends called with tensors on cuda:1 while device 0 is current run there and return there, with the
    cuda:0 bits."""
    from objectdetection_ssd_b200 import Losses, Util
    from objectdetection_ssd_b200.head import MultiboxHead, PackedGT, detect
    pri = H.priors()
    saved = Losses.ancs_xywh
    Losses.ancs_xywh = pri
    torch.cuda.set_device(0)
    try:
        def run(dev):
            r = _Round(900, pri, dev)
            tb = [torch.from_numpy(b) for b in r.gb[:16]]
            tc = [torch.from_numpy(c) for c in r.gc[:16]]
            head = MultiboxHead(pri, dev)
            out = {}
            for k, v in _head_outputs(head.loss(r.loc[:16], r.conf[:16], PackedGT(tb, tc, head.dev), True)).items():
                out[f"loss_{k}"] = v
            for k, v in _head_outputs(detect(head, r.dloc[:16], r.dconf[:16], 0.01, 0.45, 200)).items():
                out[f"det_{k}"] = v
            l = r.loc[:16].clone().requires_grad_(True)
            l1, l2 = Losses.ssd((l, r.conf[:16]), tc, tb)
            (l1 + l2).backward()
            out.update(ssd1=l1.detach(), ssd2=l2.detach(), ssd_grad=l.grad)
            for k, v in _head_outputs(Losses.inference_batch(r.dloc[:16], r.dconf[:16], 200, 0.01, 0.45)).items():
                out[f"inf_{k}"] = v
            pc = pri.to(dev)
            out["xyxy"] = Util.xywh_to_xyxy(pc)
            out["decode"] = Util.gcxgcy_to_cxcy(r.loc[0], pc)
            out["encode"] = Util.get_offsets_coords(pc, pc.flip(0))
            out["iou"] = Util.get_jaccard_tensor1(_dev(r.gb[0], dev), out["xyxy"])
            out["inter"] = Util.find_intersection(_dev(r.gb[1], dev), out["xyxy"])
            cls, obj = Util.map_prior_to_bb(out["iou"], _dev(r.gc[0], dev))
            out.update(map_cls=cls, map_obj=obj)
            db, dc, ds, gb, gc = _voc_inputs(901)
            mv = lambda xs: [x.to(dev) for x in xs]
            ap = Util.get_map(mv(db), mv(dc), mv(ds), mv(gb), mv(gc))
            torch.cuda.synchronize(dev)
            return out, ap

        got, ap1 = run(torch.device("cuda", 1))
        assert torch.cuda.current_device() == 0
        want, ap0 = run(torch.device("cuda", 0))
        for k, v in got.items():
            assert v.device == torch.device("cuda", 1), f"{k} came back on {v.device}"
            assert torch.equal(v.cpu(), want[k].cpu()), f"{k}: cuda:1 differs from cuda:0"
        assert ap1 == ap0
    finally:
        Losses.ancs_xywh = saved
        Losses._heads.clear()
