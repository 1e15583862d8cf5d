"""The host-buffer front end of the context (csrc/host_ctx.cu) at the batch sizes a training loop and the benchmark use.

``ssdhead_ctx_multibox_loss_host`` / ``_host_sparse`` split a batch into image chunks, each with its own loss-workspace
slot, its own slices of the match outputs and its own fp64 partial sums, folded by ``sum_chunks_kernel``.  Gradients come
back four ways: dense into pageable buffers (zero background written by the streaming kernel, copied back), dense into
page-locked buffers (host threads zero them chunk by chunk, the mining kernel stores its rows through UVA), packed rows
into page-locked buffers (written in place) and packed rows into pageable buffers (through device staging).  A
page-locked ``loc`` is read in place; pageable or unaligned ``loc`` is copied.  ``ssdhead_ctx_detect_host`` copies conf,
reads page-locked ``loc`` in place and takes the exhaustive or the short-list detect route by call size.

Every result here is compared bit for bit with the device step (``MultiboxHead.loss`` / ``ctx.loss_dev``) or the device
``detect`` on the same inputs; the losses, which the chunked fold adds in another order, to 1e-6 relative; and at the
benchmark's batch of 256 the batch is pinned to the float64 reference of test_gpu_trained_regime.py.  Page-locked
buffers are counted (``pinned`` below) and released as each case ends.
"""
import gc
import os
import re
import weakref

import numpy as np
import pytest
import torch

from objectdetection_ssd_b200 import ctx as CTX
from objectdetection_ssd_b200 import synth
from objectdetection_ssd_b200.pinned import PinnedBlock
from oracle import ssd_oracle as O
from tests import helpers as H
from tests.test_gpu_sharded_one_gpu import pin_full_batch
from tests.test_gpu_trained_regime import CASES, EPS, case_inputs

pytestmark = pytest.mark.gpu

C = 21
BG = C - 1
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MIN_SCORE, IOU_THR = 0.01, 0.45
PINNED_BUDGET = 1 << 30          # page-locked bytes the module may hold at once


# ----------------------------------------------------------------------------------------------------------- layout
def chunk_layout(B):
    """The image chunks of a host-buffer loss call (csrc/host_ctx.cu, loss_host_impl): (first image, images) each."""
    nchunks = min(8, max(1, B // 8))
    per = (B + nchunks - 1) // nchunks
    return [(b0, min(per, B - b0)) for b0 in range(0, B, per)]


def test_chunk_table_matches_the_source():
    with open(os.path.join(ROOT, "objectdetection_ssd_b200", "csrc", "host_ctx.cu")) as f:
        src = f.read()
    assert re.search(r"const int nchunks = std::min\(8, std::max\(1, B / 8\)\);", src)
    assert re.search(r"const int per = \(B \+ nchunks - 1\) / nchunks;", src)
    assert re.search(r"constexpr int kMaxChunks = 8;", src)
    # the chunk table is built once, by the only walk over the batch; the zeroing job, the copies and the kernels walk
    # the table, and the fold adds all of its chunks
    assert len(re.findall(r"b0 \+= per", src)) == 1
    assert re.search(r"for \(int k = 0, b0 = 0; b0 < B; \+\+k, b0 \+= per\) \{\s*const int nb = std::min\(per, B - b0\);"
                     r"\s*chunk\[k\] = \{b0, nb, \(size_t\)b0 \* P, \(size_t\)nb \* P\};", src)
    assert len(re.findall(r"for \(int k = 0; k < nchunks; \+\+k\)", src)) == 3
    assert re.search(r"sum_chunks_xchg_kernel<<<1, 1, 0, c->s_main>>>\(c->chunk_sums, nchunks,", src)
    assert re.search(r"sum_chunks_kernel<<<1, 1, 0, c->s_main>>>\(c->chunk_sums, nchunks,", src)
    assert all(len(chunk_layout(B)) == min(8, max(1, B // 8)) for B in range(1, 1025))
    # each chunk mines its own slices and workspace slot, and adds into its own partial sums
    for s in (r"c->gt_off \+ b0", r"c->npos \+ b0", r"c->cls_u8 \+ r0", r"c->chunk_sums \+ 2 \* k",
              r"\(char\*\)c->ws_loss \+ \(size_t\)k \* c->ws_loss_bytes"):
        assert re.search(s, src), s
    sizes = lambda B: [n for _, n in chunk_layout(B)]
    assert sizes(1) == [1] and sizes(7) == [7]
    assert sizes(16) == [8, 8] and sizes(256) == [32] * 8
    assert sizes(17) == [9, 8]
    assert sizes(57) == [9] * 6 + [3]
    assert sizes(65) == [9] * 7 + [2]
    assert sizes(255) == [32] * 7 + [31]


# ----------------------------------------------------------------------------------------------------------- harness
class _Pinned:
    live = 0
    peak = 0


def _account(n):
    _Pinned.live += n
    _Pinned.peak = max(_Pinned.peak, _Pinned.live)


def pinned(shape, dtype=np.float32, offset=0):
    """Page-locked array (released with its last view), counted against PINNED_BUDGET; ``offset`` bytes into its block."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape))
    blk = PinnedBlock(n * dtype.itemsize + offset)
    _account(blk.nbytes)
    weakref.finalize(blk, _account, -blk.nbytes)
    return blk.view(offset, n, dtype).reshape(shape)


@pytest.fixture(scope="module", autouse=True)
def _pinned_accounting():
    mp = pytest.MonkeyPatch()
    mp.setattr(CTX, "pinned_empty", pinned)               # SparseRows allocates through it
    yield
    mp.undo()
    print(f"\n{__name__}: peak page-locked host memory {_Pinned.peak / 2 ** 20:.0f} MiB")
    assert _Pinned.peak <= PINNED_BUDGET, f"{_Pinned.peak / 2 ** 20:.0f} MiB page-locked at once"


@pytest.fixture(autouse=True)
def _release_pinned():
    yield
    gc.collect()


_HEADS = {}


def head_for(kind="ssd300"):
    from objectdetection_ssd_b200.head import MultiboxHead
    if kind not in _HEADS:
        _HEADS[kind] = (H.priors(kind), MultiboxHead(H.priors(kind), "cuda"))
    return _HEADS[kind]


def same(a, b):
    """Identical bits (float arrays compared as their int32 patterns)."""
    a, b = np.ascontiguousarray(np.asarray(a)), np.ascontiguousarray(np.asarray(b))
    return a.shape == b.shape and np.array_equal(a.view(np.int32), b.view(np.int32))


def packed(tb, tc):
    return synth.pack_gt([b.numpy() for b in tb], [c.numpy() for c in tc])


def device_step(head, loc, conf, tb, tc):
    """The device step (flat two-kernel step) with its taps, on the host."""
    from objectdetection_ssd_b200.head import PackedGT
    o = head.loss(loc.cuda(), conf.cuda(), PackedGT(tb, tc, head.dev), with_grads=True, taps=True)
    torch.cuda.synchronize()
    return {k: v.cpu() for k, v in o.items() if torch.is_tensor(v)}


def host_inputs(loc, conf, kind="pinned"):
    """(loc, conf) host arrays: both page-locked, both pageable, page-locked conf with a page-locked loc 4 bytes into
    its block (the UVA alias is refused: not 16-byte aligned), or page-locked loc with pageable conf."""
    l, c = loc.numpy(), conf.numpy()
    if kind == "pageable":
        return l.copy(), c.copy()
    hc = c.copy() if kind == "pageable_conf" else pinned(c.shape)
    hc[...] = c
    hl = pinned(l.shape, offset=4 if kind == "offset_loc" else 0)
    hl[...] = l
    return hl, hc


MODES = ("dense_pageable", "dense_pinned", "rows_pinned", "rows_pageable")
ROW_SENTINEL = -7


def host_loss(ctx, mode, hl, hc, gt, P, cap=1024):
    """One host-buffer loss call in gradient-return `mode`; output buffers pre-filled with garbage.
    Returns (losses, dense grad_loc, dense grad_conf, rows or None)."""
    B = int(hl.shape[0])
    if mode.startswith("dense"):
        alloc = pinned if mode == "dense_pinned" else np.empty
        gl, gc_ = alloc((B, P, 4), np.float32), alloc((B, P, C), np.float32)
        gl[...] = np.nan
        gc_[...] = -3.0
        return ctx.loss_host(hl, hc, *gt, gl, gc_), gl, gc_, None
    rows = CTX.SparseRows(B, cap=cap, pinned=mode == "rows_pinned")
    rows.cnt[...] = ROW_SENTINEL
    rows.idx[...] = ROW_SENTINEL
    rows.grad_conf[...] = np.nan
    rows.grad_loc[...] = np.nan
    losses = ctx.loss_host_sparse(hl, hc, *gt, rows)
    assert int(rows.cnt[:, 0].max()) <= cap, "an image has more gradient rows than the buffers hold"
    gl, gc_ = rows.scatter(P)
    return losses, gl, gc_, rows


def check_rows(rows, d, in_place, nonzero_rows):
    """Per image: cnt = (positives + mined negatives, positives) of the device step's taps, distinct priors, positives
    first; with ``nonzero_rows`` also the non-zero rows of the dense gradients; in-place buffers untouched past the
    count."""
    B, P = d["cls_u8"].shape
    pos = d["cls_u8"].numpy() != BG
    mined = H.unpack_mask(d["mined_mask"], P).numpy()
    gl, gc_ = d["grad_loc"].numpy(), d["grad_conf"].numpy()
    for b in range(B):
        n, npos = (int(x) for x in rows.cnt[b])
        assert npos == int(pos[b].sum()) and n == npos + int(mined[b].sum()), f"image {b}: counts {n, npos}"
        if nonzero_rows:
            assert n == int((gc_[b] != 0).any(-1).sum()) and npos == int((gl[b] != 0).any(-1).sum()), f"image {b}"
        idx = rows.idx[b, :n]
        assert np.unique(idx).size == n and idx.min() >= 0 and idx.max() < P, f"image {b}: row indices"
        assert pos[b, idx[:npos]].all() and mined[b, idx[npos:]].all(), f"image {b}: positives must come first"
        if in_place:
            assert (rows.idx[b, n:] == ROW_SENTINEL).all(), f"image {b}: index written past the count"
            assert np.isnan(rows.grad_conf[b, n:]).all(), f"image {b}: conf row written past the count"
            assert np.isnan(rows.grad_loc[b, npos:]).all(), f"image {b}: loc row written past the positives"


def run_modes(ctx, pri, loc, conf, tb, tc, d, nonzero_rows=True, modes=MODES, cap=1024, kind="pinned"):
    """Every gradient-return mode on one context: gradients equal the device step's bits, losses equal across the modes
    and within 1e-6 of the device step's.  Returns the losses."""
    P = pri.shape[0]
    hl, hc = host_inputs(loc, conf, kind)
    gt = packed(tb, tc)
    got = {}
    for mode in modes:
        losses, gl, gc_, rows = host_loss(ctx, mode, hl, hc, gt, P, cap)
        assert same(gl, d["grad_loc"]), f"{mode}: grad_loc differs from the device step"
        assert same(gc_, d["grad_conf"]), f"{mode}: grad_conf differs from the device step"
        if rows is not None:
            check_rows(rows, d, mode == "rows_pinned", nonzero_rows)
        got[mode] = losses
        del gl, gc_, rows
    first = got[modes[0]]
    for mode, losses in got.items():
        assert same(np.float32(losses), np.float32(first)), f"{mode}: losses {losses} vs {modes[0]} {first}"
    dl = d["losses"].tolist()
    for a, b in zip(first, dl):
        assert abs(a - b) <= 1e-6 * abs(b), (first, dl)
    return first


def pin_host_losses(pri, loc, conf, tb, tc, d, losses):
    """The device step against the float64 reference; the host losses within their sums' budgets / (4N, N) plus one
    fp32 rounding."""
    (l1, b1), (s1, b2) = pin_full_batch(pri, loc, conf, tb, tc, d)
    N = int(d["npos"][loc.shape[0]])
    assert abs(losses[0] - l1 / (4.0 * N)) <= b1 / (4.0 * N) + EPS * abs(losses[0]), (losses[0], l1 / (4.0 * N))
    assert abs(losses[1] - s1 / N) <= b2 / N + EPS * abs(losses[1]), (losses[1], s1 / N)


# ----------------------------------------------------------------------------------------------------------- loss
@pytest.mark.parametrize("B,maxB", [(1, 1), (7, 7), (16, 16), (17, 17), (57, 57), (65, 80), (255, 255), (256, 256)])
def test_loss_host_every_mode_and_chunk_layout(B, maxB):
    """Single chunk, equal chunks, short last chunks, a context larger than the batch; at B = 256 the batch is also
    pinned to float64."""
    pri, head = head_for()
    loc, conf, tb, tc = H.train_inputs(300 + B, B, pri.shape[0])
    d = device_step(head, loc, conf, tb, tc)
    ctx = CTX.SSDHeadContext(pri.numpy(), max_batch=maxB)
    losses = run_modes(ctx, pri, loc, conf, tb, tc, d)
    ctx.close()
    if B == 256:
        pin_host_losses(pri, loc, conf, tb, tc, d, losses)


@pytest.mark.parametrize("name", ["margin_25"])
def test_loss_host_trained_head_batch_256(name):
    """A trained head's logits (zero-CE ties, mined rows whose gradient is exactly zero) at the benchmark's batch."""
    assert name in CASES
    pri, head = head_for()
    _, loc, conf, tb, tc = case_inputs(name, B=256)
    d = device_step(head, loc, conf, tb, tc)
    ctx = CTX.SSDHeadContext(pri.numpy(), max_batch=256)
    losses = run_modes(ctx, pri, loc, conf, tb, tc, d, nonzero_rows=False)
    ctx.close()
    pin_host_losses(pri, loc, conf, tb, tc, d, losses)


def test_loss_host_input_buffer_kinds():
    """Page-locked loc read in place, pageable loc, an unaligned page-locked loc (copied), pageable conf beside
    page-locked loc, and gradient buffers of mixed kinds (copy path): the same bits everywhere."""
    pri, head = head_for()
    B, P = 17, pri.shape[0]
    loc, conf, tb, tc = H.train_inputs(331, B, P)
    d = device_step(head, loc, conf, tb, tc)
    ctx = CTX.SSDHeadContext(pri.numpy(), max_batch=B)
    want = None
    for kind in ("pinned", "pageable", "offset_loc", "pageable_conf"):
        losses = run_modes(ctx, pri, loc, conf, tb, tc, d, modes=("dense_pinned", "rows_pinned", "dense_pageable"), kind=kind)
        want = want or losses
        assert losses == want, kind
    hl, hc = host_inputs(loc, conf)
    assert hl.ctypes.data % 16 == 0
    gt = packed(tb, tc)
    for gl_pinned in (True, False):
        gl = pinned((B, P, 4)) if gl_pinned else np.empty((B, P, 4), np.float32)
        gc_ = np.empty((B, P, C), np.float32) if gl_pinned else pinned((B, P, C))
        gl[...] = np.nan
        gc_[...] = np.nan
        assert ctx.loss_host(hl, hc, *gt, gl, gc_) == want
        assert same(gl, d["grad_loc"]) and same(gc_, d["grad_conf"]), f"grad_loc page-locked: {gl_pinned}"
    ctx.close()


def test_loss_host_stress_shape():
    """SSD512 priors (24 564), 60-100 gts per image, B = 128, rows up to 8192 per image: the benchmark's stress shape."""
    pri, head = head_for("ssd512")
    B = 128
    loc, conf, tb, tc = H.train_inputs(512, B, pri.shape[0], 60, 100)
    d = device_step(head, loc, conf, tb, tc)
    ctx = CTX.SSDHeadContext(pri.numpy(), max_batch=B)
    run_modes(ctx, pri, loc, conf, tb, tc, d, modes=("dense_pageable", "rows_pinned"), cap=8192)
    ctx.close()


@pytest.mark.parametrize("threads", [1, 3, 64])
def test_zero_pool_sizes(threads, monkeypatch):
    """Page-locked dense gradients with 1, 3 and 64 zeroing threads, 8 chunks with a short last one: every element the
    GPU does not write is zeroed; the pool is reused by a second, smaller batch."""
    monkeypatch.setenv("SSDHEAD_ZERO_THREADS", str(threads))
    pri, head = head_for()
    ctx = CTX.SSDHeadContext(pri.numpy(), max_batch=65)
    for B in (65, 17):
        loc, conf, tb, tc = H.train_inputs(340 + B, B, pri.shape[0])
        d = device_step(head, loc, conf, tb, tc)
        run_modes(ctx, pri, loc, conf, tb, tc, d, modes=("dense_pinned",))
    ctx.close()


# ----------------------------------------------------------------------------------------------------------- sequence
class _Dev:
    """Device tensors of one loss input set and the outputs of a device call."""

    def __init__(self, loc, conf, tb, tc):
        self.gx, self.gcl, self.off = packed(tb, tc)
        d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        self.loc, self.conf = loc.cuda(), conf.cuda()
        self.tgx, self.tgc, self.toff = d(self.gx), d(self.gcl), d(self.off)
        self.B, self.sumG = int(loc.shape[0]), int(self.off[-1])
        self.sums = torch.empty(2, dtype=torch.float64, device="cuda")
        self.losses = torch.empty(2, device="cuda")

    def args(self):
        return (self.loc.data_ptr(), self.conf.data_ptr(), self.tgx.data_ptr(), self.tgc.data_ptr(), self.toff.data_ptr(),
                self.B, self.sumG, self.sums.data_ptr(), self.losses.data_ptr())


def dev_call(ctx, x, kind, res=None):
    """loss_dev into new gradient tensors, or loss_dev_resident into ``res`` (fresh or not).  Returns host outputs."""
    st = torch.cuda.current_stream().cuda_stream
    if kind == "dev":
        gl, gc_ = torch.empty_like(x.loc), torch.empty_like(x.conf)
        ctx.loss_dev(*x.args(), gl.data_ptr(), gc_.data_ptr(), st)
    else:
        gl, gc_ = res
        ctx.loss_dev_resident(*x.args(), gl.data_ptr(), gc_.data_ptr(), st, fresh=kind == "resident_fresh")
    torch.cuda.synchronize()
    return dict(losses=x.losses.cpu(), sums=x.sums.cpu(), grad_loc=gl[:x.B].cpu(), grad_conf=gc_[:x.B].cpu())


def detect_call(ctx, hl, hc, with_prior=True):
    B, k = int(hl.shape[0]), ctx.top_k
    ob, op = np.full((B, k, 4), np.nan, np.float32), np.full((B, k), np.nan, np.float32)
    oc, oi, on = np.full((B, k), -9, np.int32), np.full((B, k), -9, np.int32), np.full((B,), -9, np.int32)
    ctx.detect_host(hl, hc, ob, op, oc, oi if with_prior else None, on, MIN_SCORE, IOU_THR)
    return dict(boxes=ob, prob=op, cls=oc, prior=oi, cnt=on)


def same_detections(a, b, keys=("boxes", "prob", "cls", "prior")):
    assert same(a["cnt"], b["cnt"]), (a["cnt"].tolist(), b["cnt"].tolist())
    for i, k in enumerate(np.asarray(a["cnt"]).tolist()):
        for key in keys:
            assert same(np.asarray(a[key][i, :k]), np.asarray(b[key][i, :k])), f"image {i}: {key}"


def test_one_context_through_a_sequence():
    """Batch sizes down and up (256, 17, 255, 1, 256) through every entry point of one context, each call equal to the
    same call on a fresh context; the pageable row staging grows from B * row_cap = 17 x (largest image's rows) to
    255 x 1024."""
    pri, head = head_for()
    P = pri.shape[0]
    ctx = CTX.SSDHeadContext(pri.numpy(), max_batch=256)
    res = (torch.full((256, P, 4), 5.0, device="cuda"), torch.full((256, P, C), -5.0, device="cuda"))
    plan = [("dense_pinned", 256), ("dev", 17), ("rows_pageable_small", 17), ("resident_fresh", 255), ("rows_pinned", 255),
            ("detect", 1), ("dense_pageable", 1), ("rows_pageable", 255), ("resident", 17), ("detect", 256), ("dev", 256),
            ("dense_pinned", 256), ("detect", 17)]
    for step, (kind, B) in enumerate(plan):
        fresh = CTX.SSDHeadContext(pri.numpy(), max_batch=B)
        what = f"step {step} ({kind}, B={B})"
        if kind == "detect":
            loc, conf = H.detect_inputs(360 + step, B, P)
            hl, hc = host_inputs(loc, conf)
            same_detections(detect_call(ctx, hl, hc), detect_call(fresh, hl, hc))
        elif kind in ("dev", "resident", "resident_fresh"):
            x = _Dev(*H.train_inputs(360 + step, B, P))
            got = dev_call(ctx, x, kind, res)
            fres = (torch.empty_like(x.loc), torch.empty_like(x.conf))
            want = dev_call(fresh, x, "dev" if kind == "dev" else "resident_fresh", fres)
            for key in want:
                assert same(got[key].numpy(), want[key].numpy()), f"{what}: {key}"
        else:
            loc, conf, tb, tc = H.train_inputs(360 + step, B, P)
            hl, hc = host_inputs(loc, conf)
            gt = packed(tb, tc)
            mode, cap = kind, 1024
            if kind == "rows_pageable_small":
                probe = CTX.SSDHeadContext(pri.numpy(), max_batch=B)
                _, _, _, rows = host_loss(probe, "rows_pinned", hl, hc, gt, P)
                probe.close()
                mode, cap = "rows_pageable", int(rows.cnt[:, 0].max())
                assert 255 * 1024 > B * cap
            a = host_loss(ctx, mode, hl, hc, gt, P, cap)
            b = host_loss(fresh, mode, hl, hc, gt, P, cap)
            assert same(np.float32(a[0]), np.float32(b[0])), f"{what}: losses {a[0]} vs {b[0]}"
            assert same(a[1], b[1]) and same(a[2], b[2]), f"{what}: gradients"
            if a[3] is not None:
                assert same(a[3].cnt, b[3].cnt), f"{what}: row counts"
        fresh.close()
    ctx.close()


# ----------------------------------------------------------------------------------------------------------- ordering
SLEEP_CYCLES = 200_000_000       # ~100 ms at the B200's clock; a host call of 4 images takes a few ms


@pytest.mark.parametrize("call", ["loss_host", "loss_host_sparse", "detect_host"])
def test_host_call_waits_for_the_pending_device_step(call):
    """A device step queued behind ~100 ms of other work on the caller's stream, then at once a host call on the same
    context: the host call must order itself after the device step (which uses the same match outputs and workspace),
    so when it returns the caller's stream is idle.  Both results are checked after a synchronize.  The host call
    cannot overlap the device step either way: it finishes long before the queued work would reach the device step."""
    pri, head = head_for()
    P = pri.shape[0]
    x = _Dev(*H.train_inputs(370, 16, P))
    loc, conf, tb, tc = H.train_inputs(371, 4, P)
    hl, hc = host_inputs(loc, conf)
    gt = packed(tb, tc)
    ref = CTX.SSDHeadContext(pri.numpy(), max_batch=16)
    want_dev = dev_call(ref, x, "dev")

    def host(c):
        if call == "detect_host":
            return detect_call(c, hl, hc)
        return host_loss(c, "dense_pinned" if call == "loss_host" else "rows_pinned", hl, hc, gt, P)

    want_host = host(ref)
    ref.close()
    ctx = CTX.SSDHeadContext(pri.numpy(), max_batch=16)
    host(ctx)                                            # warm: zeroing threads started, buffers in place
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    gl, gc_ = torch.empty_like(x.loc), torch.empty_like(x.conf)
    torch.cuda._sleep(SLEEP_CYCLES)
    ctx.loss_dev(*x.args(), gl.data_ptr(), gc_.data_ptr(), stream.cuda_stream)
    got_host = host(ctx)
    idle = stream.query()
    torch.cuda.synchronize()
    assert idle, f"{call} returned while the device step queued before it on the same context was still pending"
    assert same(x.losses.cpu().numpy(), want_dev["losses"].numpy()) and same(x.sums.cpu().numpy(), want_dev["sums"].numpy())
    assert same(gl.cpu().numpy(), want_dev["grad_loc"].numpy()) and same(gc_.cpu().numpy(), want_dev["grad_conf"].numpy())
    if call == "detect_host":
        same_detections(got_host, want_host)
    else:
        assert got_host[0] == want_host[0]
        assert same(got_host[1], want_host[1]) and same(got_host[2], want_host[2])
    ctx.close()


def test_host_call_after_a_captured_device_step():
    """A captured context step records nothing the host calls wait on (an event recorded inside a capture cannot be
    waited on from outside it): after the replay is synchronized, a host call on the same context runs and is right."""
    pri, head = head_for()
    P = pri.shape[0]
    x = _Dev(*H.train_inputs(380, 8, P))
    loc, conf, tb, tc = H.train_inputs(381, 4, P)
    hl, hc = host_inputs(loc, conf)
    gt = packed(tb, tc)
    ref = CTX.SSDHeadContext(pri.numpy(), max_batch=8)
    want_dev = dev_call(ref, x, "dev")
    want_host = host_loss(ref, "dense_pinned", hl, hc, gt, P)
    ref.close()
    ctx = CTX.SSDHeadContext(pri.numpy(), max_batch=8)
    gl, gc_ = torch.empty_like(x.loc), torch.empty_like(x.conf)
    ctx.loss_dev(*x.args(), gl.data_ptr(), gc_.data_ptr(), torch.cuda.current_stream().cuda_stream)     # eager first
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ctx.loss_dev(*x.args(), gl.data_ptr(), gc_.data_ptr(), torch.cuda.current_stream().cuda_stream)
    gl.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert same(gl.cpu().numpy(), want_dev["grad_loc"].numpy()) and same(gc_.cpu().numpy(), want_dev["grad_conf"].numpy())
    got = host_loss(ctx, "dense_pinned", hl, hc, gt, P)
    assert got[0] == want_host[0] and same(got[1], want_host[1]) and same(got[2], want_host[2])
    del g
    ctx.close()


# ----------------------------------------------------------------------------------------------------------- detect
def test_detect_route_threshold_matches_the_source():
    with open(os.path.join(ROOT, "objectdetection_ssd_b200", "csrc", "detect.cu")) as f:
        src = f.read()
    assert "return (long long)B * P >= 900000;" in src
    P = H.priors().shape[0]
    assert 103 * P < 900000 <= 104 * P


def device_detect(head, loc, conf, top_k):
    from objectdetection_ssd_b200.head import detect
    out = detect(head, loc, conf, MIN_SCORE, IOU_THR, top_k)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def check_detect_host(ctx, head, loc, conf, kind="pinned"):
    """detect_host (with and without out_prior) equals the device detect with the context's top_k, bit for bit."""
    hl, hc = host_inputs(loc, conf, kind)
    want = device_detect(head, loc, conf, ctx.top_k)
    got = detect_call(ctx, hl, hc)
    same_detections(got, want)
    same_detections(detect_call(ctx, hl, hc, with_prior=False), want, keys=("boxes", "prob", "cls"))
    return got


@pytest.mark.parametrize("B,kind", [(64, "pinned"), (64, "offset_loc"), (103, "pinned"), (104, "pinned"),
                                    (104, "offset_loc"), (256, "pinned"), (256, "pageable")])
def test_detect_host_equals_device_detect(B, kind, monkeypatch):
    """Exhaustive route up to B = 103, short list from B = 104 (SSD300); page-locked loc read in place by either route,
    pageable or unaligned loc copied.  At B = 256 a sample of images against the oracle."""
    monkeypatch.delenv("SSDHEAD_DETECT_SHORTLIST", raising=False)
    pri, head = head_for()
    loc, conf = H.detect_inputs(390 + B, B, pri.shape[0])
    ctx = CTX.SSDHeadContext(pri.numpy(), max_batch=B)
    got = check_detect_host(ctx, head, loc, conf, kind)
    ctx.close()
    assert (got["cnt"] == 200).all()
    if B == 256 and kind == "pinned":
        out = {k: torch.from_numpy(v) for k, v in got.items()}
        H.compare_detect_with_oracle(out, loc, conf, pri, MIN_SCORE, IOU_THR, 200, [0, 101, 202, 255])


@pytest.mark.parametrize("top_k", [1, 400])
def test_detect_host_top_k(top_k, monkeypatch):
    monkeypatch.delenv("SSDHEAD_DETECT_SHORTLIST", raising=False)
    pri, head = head_for()
    ctx = CTX.SSDHeadContext(pri.numpy(), max_batch=104, top_k=top_k)
    for B in (104, 9):
        loc, conf = H.detect_inputs(395 + B, B, pri.shape[0])
        got = check_detect_host(ctx, head, loc, conf)
        assert (got["cnt"] > 0).all() and (got["cnt"] <= top_k).all()
        assert top_k > 1 or (got["cnt"] == 1).all()
    ctx.close()


def test_detect_host_with_images_on_the_exact_fallback(monkeypatch):
    """Every fourth image of a short-list batch holds 40 box sites in two classes (heavy suppression): the short list
    cannot decide those images and their sweep lists them again in full.  The host call equals the device detect."""
    from objectdetection_ssd_b200.head import detect_fallbacks
    from tests.test_gpu_detect_shortlist import _few_sites_inputs
    monkeypatch.delenv("SSDHEAD_DETECT_SHORTLIST", raising=False)
    pri, head = head_for()
    B, P = 104, pri.shape[0]
    loc, conf = H.detect_inputs(398, B, P)
    boxes, probs = _few_sites_inputs(399, 4, P, classes=(2, 11))
    heavy = list(range(1, B, 4))
    for j, i in enumerate(heavy):
        loc[i] = O.encode(boxes[j % 4], pri)
        conf[i] = torch.log(probs[j % 4].clamp_min(1e-12))
    ctx = CTX.SSDHeadContext(pri.numpy(), max_batch=B)
    got = check_detect_host(ctx, head, loc, conf)
    # the context exposes no fallback count: the device detect's count shows these inputs take the fallback, and the
    # host call's bit equality with the device detect (check_detect_host) shows it produced the same output
    assert detect_fallbacks(head, B) == len(heavy)
    assert (got["cnt"][heavy] < 200).all() and (np.delete(got["cnt"], heavy) == 200).all()
    ctx.close()
