"""Host-side operator layer over libssdhead.so: device buffers, streams and autograd plumbing.

PyTorch is used here only for device memory, the current CUDA stream, autograd wiring and
(optionally) ``torch.distributed``; all arithmetic of the path runs in the CUDA kernels of
``csrc/`` reached through the C ABI (``include/ssdhead.h``).  There is no CPU fallback: every
entry point raises if the tensors cannot be placed on a CUDA device or the library is missing.

Reference call sites this layer serves: ``ssd`` (Losses.py:119-134), ``ssd1_`` (Losses.py:136-199),
``map_prior_to_bb`` (Util.py:333-352), ``inference`` (Losses.py:11-98).
"""
from __future__ import annotations

import threading
from contextlib import contextmanager
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from .priors import cxcywh_to_xyxy_host

POS_IOU = 0.5      # Losses.py:171
NEG_RATIO = 3      # Losses.py:189


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream(dev: torch.device):
    return torch.cuda.current_stream(dev).cuda_stream


def require_cuda(dev) -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("objectdetection_ssd_b200: no CUDA device - the SSD head path has no CPU fallback")
    dev = torch.device(dev)
    if dev.type != "cuda":
        raise RuntimeError(f"objectdetection_ssd_b200: expected a CUDA device, got {dev}")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev


_staging_pool = None     # pinned.StagingPool, created with the first host-list batch
_staging_pool_lock = threading.Lock()


def refuse_capture(what: str) -> None:
    """Raise if the current stream is capturing a CUDA graph: ``what`` packs its gts from host values and shares
    workspaces between calls, so a graph of it would replay stale gts or write into freed memory."""
    if torch.cuda.is_available() and torch.cuda.is_current_stream_capturing():
        raise RuntimeError(f"{what} cannot be captured into a CUDA graph (it reads its gt count on the host and shares "
                           "its workspaces); use objectdetection_ssd_b200.Losses.StaticHead: load() the gts before "
                           "each replay, capture StaticHead.loss / loss_levels / detect")


class PackedGT:
    """Ragged gt lists packed once: boxes [sumG,4] f32, classes [sumG] f32, offsets int32 [B+1]
    (host-side equivalent of Losses.py:129-130; no per-image synchronisation).

    This sits on the per-step path of ``ssd()`` (train_function.py:62-63,82), so the per-image Python work is kept to
    one shape read: the lists are concatenated by ONE ``torch.cat`` each - for host lists straight into a recycled
    page-locked block that then crosses to the device in one copy, offsets included."""

    def __init__(self, boxes: Sequence[torch.Tensor], classes: Sequence[torch.Tensor], dev: torch.device):
        refuse_capture("PackedGT")
        try:
            counts = [b.shape[0] for b in boxes]
        except IndexError:                       # a 0-dim entry: no box
            counts = [b.shape[0] if b.dim() > 0 else 0 for b in boxes]
        if 0 in counts:
            # the reference fails the same way on an image without objects (Losses.py:153, max over an empty dim)
            raise IndexError(f"image {counts.index(0)} has no ground-truth box: max() over an empty dimension")
        self.B = len(counts)
        if len(classes) != self.B:
            raise ValueError(f"{self.B} box lists but {len(classes)} class lists")
        offs = np.zeros(self.B + 1, dtype=np.int32)
        if self.B:
            np.cumsum(counts, out=offs[1:])
        self._off_np = offs
        self.sumG = int(offs[-1])
        self.maxG = max(counts) if counts else 0
        cuda = torch.cuda.is_available()
        b0, c0 = (boxes[0], classes[0]) if self.B else (None, None)
        if cuda and self.B and b0.device.type == "cpu" and c0.device.type == "cpu":
            # host lists (what a DataLoader hands over): concatenated straight into a recycled page-locked block (no
            # cudaHostAlloc / cudaFreeHost per step), ONE copy of the block to the device; the block returns to the pool
            # behind an event recorded after the copy, so it is never rewritten while the DMA engine may still read it
            global _staging_pool
            if _staging_pool is None:
                from .pinned import StagingPool
                with _staging_pool_lock:
                    if _staging_pool is None:
                        _staging_pool = StagingPool()
            from .pinned import gt_layout
            st = _staging_pool.acquire(self.sumG, self.B)
            try:
                self._fill_staging(st, boxes, classes)
            except Exception:
                _staging_pool.release(st, st.event)
                raise
            blk = torch.empty(st.nbytes, dtype=torch.uint8, device=dev)
            blk.copy_(st.raw_t, non_blocking=True)
            if st.event is None or st.event_dev != dev:         # an event is recorded on streams of one device only
                st.event, st.event_dev = torch.cuda.Event(), dev
            st.event.record(torch.cuda.current_stream(dev))
            _staging_pool.release(st, st.event)
            o0, o1, o2, _ = gt_layout(st.capacity, self.B)
            self.boxes = blk[o0:o0 + self.sumG * 16].view(torch.float32).view(self.sumG, 4)
            self.classes = blk[o1:o1 + self.sumG * 4].view(torch.float32)
            self.off = blk[o2:o2 + (self.B + 1) * 4].view(torch.int32)
            return
        self.boxes = self._cat(boxes, 4).to(device=dev, dtype=torch.float32)
        self.classes = self._cat(classes, 0).to(device=dev, dtype=torch.float32)
        if self.boxes.shape[0] != self.sumG or self.classes.shape[0] != self.sumG:
            raise ValueError(f"gt lists disagree: {self.boxes.shape[0]} boxes, {self.classes.shape[0]} classes, {self.sumG} expected")
        self.off = torch.from_numpy(offs).pin_memory().to(dev, non_blocking=True) if cuda else torch.from_numpy(offs)

    @staticmethod
    def _cat(tensors, width):
        """One concatenation; tensors of unexpected rank (e.g. a single box given as [4]) are reshaped first."""
        want = 2 if width else 1
        if all(t.dim() == want for t in tensors[:1]):
            try:
                return torch.cat(list(tensors))
            except RuntimeError:
                pass
        return torch.cat([t.reshape(-1, width) if width else t.reshape(-1) for t in tensors])

    @property
    def off_host(self):
        """Offsets as a Python list (tests, debug taps)."""
        return self._off_np.tolist()

    def _fill_staging(self, st, boxes, classes):
        _staging_views(st)
        n = self.sumG
        # one concatenation per list, then one small copy into the block (copy_ converts int64 class ids and checks the
        # shapes: [n,4] boxes, [n] classes)
        st.boxes_t[:n].copy_(self._cat(boxes, 4))
        st.classes_t[:n].copy_(self._cat(classes, 0))
        st.offsets[:] = self._off_np


def _staging_views(st):
    """torch views of a staging block's pinned arrays, made once per block."""
    if getattr(st, "boxes_t", None) is None:
        st.boxes_t = torch.from_numpy(st.boxes)
        st.classes_t = torch.from_numpy(st.classes)
        st.offsets_t = torch.from_numpy(st.offsets)
        st.raw_t = torch.from_numpy(st.raw)


class MultiboxHead:
    """Prior tables and workspaces of one CUDA device.

    One head may be used from several streams and host threads: every library call runs under the head's lock, on the
    head's device, and waits for the last use of each workspace it takes when that use was on another stream."""

    _ordered = True          # calls on different streams are ordered on the workspaces (see _calls)

    def __init__(self, priors_cxcywh: torch.Tensor, device=None, num_classes: int = 21):
        self.dev = require_cuda(device if device is not None else "cuda")
        self.lib = _lib.load()
        pc = priors_cxcywh.detach().to("cpu", torch.float32).contiguous()
        self.P = int(pc.shape[0])
        self.C = int(num_classes)
        self.pri_cxcywh = pc.to(self.dev)
        self.pri_xyxy = cxcywh_to_xyxy_host(pc).to(self.dev)     # same fp32 ops as Util.py:93-96
        self._ws = {}
        self._ws_need = {}
        self._ws_last = {}       # which -> (event recorded behind the workspace's last use, id of that use's stream)
        self._lock = threading.RLock()

    # ------------------------------------------------------------------ workspaces
    @contextmanager
    def _calls(self, *specs):
        """Context of one or more library calls: this head's lock and device, and the workspaces ``specs`` (``(which, B,
        n)`` each, as ``_workspace`` takes them) ready for the current stream.  One event recorded behind the calls marks
        the new last use of those workspaces, so a later call on another stream (or from another thread) waits for it
        before it grows, re-zeroes or uses one of them."""
        with self._lock, torch.cuda.device(self.dev):
            bufs = [self._workspace(*sp) for sp in specs]
            try:
                yield bufs
            finally:
                if specs and self._ordered:
                    cur = torch.cuda.current_stream(self.dev)
                    ev = torch.cuda.Event()
                    ev.record(cur)
                    for sp in specs:
                        self._ws_last[sp[0]] = (ev, cur.cuda_stream)

    def _workspace(self, which: int, B: int, n: int) -> torch.Tensor:
        # sized for n rounded up to a multiple of 1024 (the gt count changes every training step; a larger buffer is
        # always accepted), so the size query leaves the per-step path
        nq = (n + 1023) // 1024 * 1024 if n > 0 else 0
        need = self._ws_need.get((which, B, nq))
        if need is None:
            need = int(self.lib.ssdhead_workspace_bytes(which, B, self.P, self.C, nq))
            self._ws_need[(which, B, nq)] = need
        if need == 0:
            raise RuntimeError("ssdhead: unsupported shape for this entry point "
                               f"(B={B}, P={self.P}, C={self.C})")
        # Every kernel leaves every counter it used zeroed again and writes the other regions before it reads them, so
        # a buffer that was zero-filled once stays valid when only the gt count `n` changes (it does on every training
        # step).  A change of the batch size is re-zeroed anyway - it is rare and keeps the header's contract
        # (include/ssdhead.h, "re-zero a buffer before reusing it with another shape") to the letter.
        # On another stream than its last use, the current stream first waits for that use: the zero-fill, the replacement and
        # the call are then ordered after it.  A buffer used on a stream other than the one that allocated it is recorded on
        # that stream, so the caching allocator does not hand its memory out again before that stream is done with it.
        key = B
        st = torch.cuda.current_stream(self.dev)
        used = self._ws_last.get(which)
        if used is not None and used[1] != st.cuda_stream:
            st.wait_event(used[0])
        cur, last, home = self._ws.get(which, (None, None, None))
        if cur is None or cur.numel() < need:
            with torch.cuda.device(self.dev):
                cur = torch.zeros(max(need, 2 * (cur.numel() if cur is not None else 0)) + 4096, dtype=torch.uint8,
                                  device=self.dev)
            home = st.cuda_stream
        elif last != key:
            cur.zero_()
        if st.cuda_stream != home:
            cur.record_stream(st)
        self._ws[which] = (cur, key, home)
        return cur

    def _dense_f32(self, t: torch.Tensor) -> torch.Tensor:
        """fp32, dense, on this device - without a torch call in the common case."""
        if t.dtype == torch.float32 and t.device == self.dev and t.is_contiguous():
            return t
        return t.detach().to(device=self.dev, dtype=torch.float32).contiguous()

    # ------------------------------------------------------------------ match
    def _match_outputs(self, gt: PackedGT, want_maps: bool):
        B = gt.B
        outs = dict(best_prior=torch.empty(max(gt.sumG, 1), dtype=torch.int32, device=self.dev),
                    npos=torch.empty(B + 1, dtype=torch.int32, device=self.dev),
                    cls_u8=torch.empty(B, self.P, dtype=torch.uint8, device=self.dev), obj=None, cls=None)
        if want_maps:
            outs["obj"] = torch.empty(B, self.P, dtype=torch.int32, device=self.dev)
            outs["cls"] = torch.empty(B, self.P, dtype=torch.int32, device=self.dev)
        return outs

    def match(self, gt: PackedGT, want_maps: bool = False, pos_iou: float = POS_IOU, outs=None):
        """Losses.py:150-171.  Returns dict(best_prior, npos[B+1], cls_u8[B,P], obj[B,P]|None, cls[B,P]|None)."""
        B = gt.B
        o = outs if outs is not None else self._match_outputs(gt, want_maps)
        with self._calls((_lib.WS_MATCH, B, gt.sumG)) as (ws,):
            _lib.check(self.lib.ssdhead_match(
                _ptr(gt.boxes), _ptr(gt.classes), _ptr(gt.off), _ptr(self.pri_xyxy),
                B, self.P, self.C, gt.sumG, pos_iou,
                _ptr(o["best_prior"]), _ptr(o["npos"]), _ptr(o["cls_u8"]), _ptr(o["obj"]), _ptr(o["cls"]),
                _ptr(ws), ws.numel(), _stream(self.dev)), "ssdhead_match")
        return o

    # ------------------------------------------------------------------ loss
    def loss(self, loc: torch.Tensor, conf: torch.Tensor, gt: PackedGT, with_grads: bool,
             neg_ratio: int = NEG_RATIO, pos_iou: float = POS_IOU, taps: bool = False,
             group=None, match=None):
        """Losses.py:119-199 on device.  Returns dict(losses[2], sums[2], npos, grad_loc, grad_conf, ...).

        ``group``: a torch.distributed process group over which the batch is sharded by image;
        the positive count is all-reduced before the loss kernel (it scales the gradients) and
        the loss sums after it (SURVEY.md section 8(e))."""
        B, P, C = int(loc.shape[0]), self.P, self.C
        if tuple(loc.shape) != (B, P, 4) or tuple(conf.shape) != (B, P, C) or gt.B != B:
            raise ValueError(f"expected loc [B,{P},4] and conf [B,{P},{C}] with B gt lists, got "
                             f"{tuple(loc.shape)}, {tuple(conf.shape)}, {gt.B}")
        loc = self._dense_f32(loc)
        conf = self._dense_f32(conf)
        sums = torch.empty(2, dtype=torch.float64, device=self.dev)
        losses = torch.empty(2, dtype=torch.float32, device=self.dev)
        grad_loc = grad_conf = mined = ce = None
        if with_grads:
            grad_loc = torch.empty_like(loc)
            grad_conf = torch.empty_like(conf)
        if taps:
            mined = torch.empty(B, (P + 31) // 32, dtype=torch.int32, device=self.dev)
            ce = torch.empty(B, P, dtype=torch.float32, device=self.dev)
        m = match
        specs = [(_lib.WS_LOSS, B, 0)] + ([(_lib.WS_MATCH, B, gt.sumG)] if m is None else [])
        with self._calls(*specs) as wss:
            return self._loss_calls(loc, conf, gt, B, P, C, neg_ratio, pos_iou, group, m, wss, sums, losses, grad_loc,
                                    grad_conf, mined, ce)

    def _loss_calls(self, loc, conf, gt, B, P, C, neg_ratio, pos_iou, group, m, wss, sums, losses, grad_loc, grad_conf,
                    mined, ce):
        ws, wm = wss[0], (wss[1] if len(wss) > 1 else None)
        cur = torch.cuda.current_stream(self.dev)
        if m is None and group is None:
            # hot path, one GPU: two kernels (streaming CE + fused natural match; mining + fused forced-match finaliser)
            m = self._match_outputs(gt, False)
            _lib.check(self.lib.ssdhead_multibox_step(
                _ptr(loc), _ptr(conf), _ptr(gt.boxes), _ptr(gt.classes), _ptr(gt.off),
                _ptr(self.pri_xyxy), _ptr(self.pri_cxcywh), B, P, C, gt.sumG, int(neg_ratio), float(pos_iou),
                _ptr(sums), _ptr(losses), _ptr(grad_loc), _ptr(grad_conf),
                _ptr(m["cls_u8"]), _ptr(m["best_prior"]), _ptr(m["npos"]), _ptr(mined), _ptr(ce),
                _ptr(ws), ws.numel(), _ptr(wm), wm.numel(), cur.cuda_stream), "ssdhead_multibox_step")
            npos = m["npos"]
            return dict(losses=losses, sums=sums, npos=npos, npos_norm=npos[B:B + 1], grad_loc=grad_loc,
                        grad_conf=grad_conf, mined_mask=mined, ce=ce, best_prior=m["best_prior"], cls_u8=m["cls_u8"])
        if m is None:
            # sharded batch: the natural match rides inside the CE streaming kernel, a small finaliser applies the
            # forced-match override; the positive count is all-reduced before the mining kernel
            m = self._match_outputs(gt, False)
            _lib.check(self.lib.ssdhead_ce_match_stream(
                _ptr(conf), _ptr(gt.boxes), _ptr(gt.classes), _ptr(gt.off), _ptr(self.pri_xyxy),
                B, P, C, gt.sumG, float(pos_iou), _ptr(ce), _ptr(grad_loc), _ptr(grad_conf),
                _ptr(m["cls_u8"]), _ptr(m["best_prior"]), _ptr(m["npos"]),
                _ptr(ws), ws.numel(), _ptr(wm), wm.numel(), 1, cur.cuda_stream), "ssdhead_ce_match_stream")
        else:
            # a match computed beforehand with ssdhead_match (e.g. with the debug taps)
            _lib.check(self.lib.ssdhead_ce_stream(
                _ptr(conf), B, P, C, _ptr(ce), _ptr(grad_loc), _ptr(grad_conf),
                _ptr(ws), ws.numel(), cur.cuda_stream), "ssdhead_ce_stream")
        npos = m["npos"]
        npos_norm = npos[B:B + 1]
        if group is not None:
            import torch.distributed as dist
            npos_norm = npos_norm.clone()
            dist.all_reduce(npos_norm, op=dist.ReduceOp.SUM, group=group)
        _lib.check(self.lib.ssdhead_mine(
            _ptr(loc), _ptr(conf), _ptr(gt.boxes), _ptr(gt.classes), _ptr(gt.off),
            _ptr(self.pri_xyxy), _ptr(self.pri_cxcywh),
            _ptr(m["best_prior"]), _ptr(npos), _ptr(npos_norm), _ptr(m["cls_u8"]),
            B, P, C, int(neg_ratio), float(pos_iou),
            _ptr(sums), _ptr(losses), _ptr(grad_loc), _ptr(grad_conf), _ptr(mined), _ptr(ce),
            _ptr(ws), ws.numel(), cur.cuda_stream), "ssdhead_mine")
        if group is not None:
            import torch.distributed as dist
            dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
            _lib.check(self.lib.ssdhead_finish_loss(_ptr(sums), _ptr(npos_norm), _ptr(losses),
                                                    _stream(self.dev)), "ssdhead_finish_loss")
        return dict(losses=losses, sums=sums, npos=npos, npos_norm=npos_norm, grad_loc=grad_loc,
                    grad_conf=grad_conf, mined_mask=mined, ce=ce, best_prior=m["best_prior"], cls_u8=m["cls_u8"])

    # ------------------------------------------------------------------ per-level head tensors (SURVEY 8(f) #3)
    def _levels(self, loc_levels, conf_levels, grads=None):
        """Validate per-level tensors ([B, n_l, 4] / [B, n_l, C], e.g. NHWC conv outputs viewed as rows) and build the
        ``ssdhead_levels`` struct.  Returns (struct, loc list, conf list, B) - the lists keep the tensors alive."""
        L = len(conf_levels)
        if L < 1 or L > _lib.MAX_LEVELS or len(loc_levels) != L:
            raise ValueError(f"expected 1..{_lib.MAX_LEVELS} levels with one loc and one conf tensor each")
        B = int(conf_levels[0].shape[0])
        locs, confs = [], []
        def rows(t, width):
            # the common case (fp32, on this device, dense) costs no torch call beyond the view
            if not (t.dtype == torch.float32 and t.device == self.dev and t.is_contiguous()):
                t = t.to(device=self.dev, dtype=torch.float32).contiguous()
            return t.detach().view(B, -1, width)

        for lo, co in zip(loc_levels, conf_levels):
            lo, co = rows(lo, 4), rows(co, self.C)
            if lo.shape[1] != co.shape[1]:
                raise ValueError(f"level with {lo.shape[1]} loc rows but {co.shape[1]} conf rows")
            locs.append(lo)
            confs.append(co)
        if sum(int(c.shape[1]) for c in confs) != self.P:
            raise ValueError(f"levels hold {sum(int(c.shape[1]) for c in confs)} priors per image, the prior table {self.P}")
        st = _lib.Levels()
        st.num_levels = L
        for i in range(L):
            st.count[i] = int(confs[i].shape[1])
            st.conf[i] = confs[i].data_ptr()
            st.loc[i] = locs[i].data_ptr()
            st.grad_conf[i] = grads[1][i].data_ptr() if grads else None
            st.grad_loc[i] = grads[0][i].data_ptr() if grads else None
        return st, locs, confs, B

    def loss_levels(self, loc_levels, conf_levels, gt: PackedGT, with_grads: bool,
                    neg_ratio: int = NEG_RATIO, pos_iou: float = POS_IOU):
        """``loss`` on per-level tensors (no concatenated [B,P,*] tensor in either direction): same two kernels,
        bit-identical results; gradients come back as per-level lists in the layout of the inputs."""
        B0 = int(conf_levels[0].shape[0])
        grads = None
        if with_grads:
            grads = ([torch.empty(B0, int(c.shape[1]) if c.dim() == 3 else c.numel() // (B0 * self.C), 4, device=self.dev)
                      for c in conf_levels],
                     [torch.empty(B0, int(c.shape[1]) if c.dim() == 3 else c.numel() // (B0 * self.C), self.C, device=self.dev)
                      for c in conf_levels])
        st, locs, confs, B = self._levels(loc_levels, conf_levels, grads)
        if gt.B != B:
            raise ValueError(f"{B} images but {gt.B} gt lists")
        sums = torch.empty(2, dtype=torch.float64, device=self.dev)
        losses = torch.empty(2, dtype=torch.float32, device=self.dev)
        m = self._match_outputs(gt, False)
        import ctypes
        with self._calls((_lib.WS_LOSS, B, 0), (_lib.WS_MATCH, B, gt.sumG)) as (ws, wm):
            _lib.check(self.lib.ssdhead_multibox_step_levels(
                ctypes.addressof(st), _ptr(gt.boxes), _ptr(gt.classes), _ptr(gt.off),
                _ptr(self.pri_xyxy), _ptr(self.pri_cxcywh), B, self.P, self.C, gt.sumG, int(neg_ratio), float(pos_iou),
                _ptr(sums), _ptr(losses), _ptr(m["cls_u8"]), _ptr(m["best_prior"]), _ptr(m["npos"]),
                _ptr(ws), ws.numel(), _ptr(wm), wm.numel(), _stream(self.dev)), "ssdhead_multibox_step_levels")
        return dict(losses=losses, sums=sums, npos=m["npos"], grad_loc=grads[0] if grads else None,
                    grad_conf=grads[1] if grads else None, best_prior=m["best_prior"], cls_u8=m["cls_u8"],
                    _keep=(locs, confs))

    def scale_grads(self, grad_loc: torch.Tensor, grad_conf: torch.Tensor, gout: torch.Tensor):
        with self._calls():
            _lib.check(self.lib.ssdhead_scale_grads(_ptr(grad_loc), grad_loc.numel(), _ptr(grad_conf),
                                                    grad_conf.numel(), _ptr(gout), _stream(self.dev)),
                       "ssdhead_scale_grads")


def _upstream(head, g_loc_loss, g_conf_loss) -> torch.Tensor:
    """The two upstream gradients as one fp32 [2] device tensor (read by the scale kernel on the device: no sync)."""
    if g_loc_loss is None or g_conf_loss is None:
        z = torch.zeros((), dtype=torch.float32, device=head.dev)
        g_loc_loss = z if g_loc_loss is None else g_loc_loss
        g_conf_loss = z if g_conf_loss is None else g_conf_loss
    gout = torch.stack((g_loc_loss.reshape(()), g_conf_loss.reshape(())))
    if gout.dtype != torch.float32 or gout.device != head.dev:
        gout = gout.to(head.dev, torch.float32)
    return gout


class _MultiboxLossFn(torch.autograd.Function):
    """Autograd node for ``ssd()``: the forward kernel already wrote the gradients for unit upstream
    gradients; backward rescales them on the device only if the upstream gradients are not 1."""

    @staticmethod
    def forward(ctx, loc, conf, head: MultiboxHead, gt: PackedGT, neg_ratio, pos_iou, group, need):
        # `need` is decided by the caller: inside forward() grad mode is always off and ctx.needs_input_grad is set even
        # under torch.no_grad(), so a validation loop would otherwise pay for 0.23 GB of dense gradients per step
        out = head.loss(loc, conf, gt, with_grads=need, neg_ratio=neg_ratio, pos_iou=pos_iou, group=group)
        ctx.head = head
        ctx.src = (loc.device, conf.device, loc.dtype, conf.dtype)
        ctx.grads = (out["grad_loc"], out["grad_conf"])
        a, b = out["losses"].unbind(0)          # views of a tensor made in this call: no copy kernels
        return a, b

    @staticmethod
    def backward(ctx, g_loc_loss, g_conf_loss):
        if ctx.grads is None or ctx.grads[0] is None:
            raise RuntimeError("ssd(): backward called twice (or without grad-requiring inputs); the fused "
                               "kernel frees its gradient buffers after the first backward, as autograd does")
        gl, gc = ctx.grads
        ctx.grads = None
        head = ctx.head
        head.scale_grads(gl, gc, _upstream(head, g_loc_loss, g_conf_loss))
        ld, cd, lt, ct = ctx.src
        if ld == gl.device and lt == gl.dtype and cd == gc.device and ct == gc.dtype:
            return gl, gc, None, None, None, None, None, None
        return gl.to(device=ld, dtype=lt), gc.to(device=cd, dtype=ct), None, None, None, None, None, None


def multibox_loss(head: MultiboxHead, loc: torch.Tensor, conf: torch.Tensor,
                  gt_boxes: List[torch.Tensor], gt_classes: List[torch.Tensor],
                  neg_ratio: int = NEG_RATIO, pos_iou: float = POS_IOU, group=None):
    """(loc_loss, conf_loss) as 0-dim tensors with grad_fn - the return of ``ssd()`` (Losses.py:134)."""
    gt = PackedGT(gt_boxes, gt_classes, head.dev)
    need = torch.is_grad_enabled() and (loc.requires_grad or conf.requires_grad)
    return _MultiboxLossFn.apply(loc, conf, head, gt, neg_ratio, pos_iou, group, need)


def _detect(head: MultiboxHead, a: torch.Tensor, b: torch.Tensor, min_score: float, iou_thr: float, top_k: int,
            img_wh: Optional[torch.Tensor], max_candidates: int, from_scores: bool):
    """inference() over a batch (Losses.py:11-98).  ``a, b`` = (loc, conf) or, stage-isolated, (boxes_cxcywh, probs).
    Returns dict(boxes [B,top_k,4], prob [B,top_k], cls int32, prior int32, cnt int32 [B])."""
    B, P, C = int(a.shape[0]), head.P, head.C
    if tuple(a.shape) != (B, P, 4) or tuple(b.shape) != (B, P, C):
        raise ValueError(f"expected [B,{P},4] and [B,{P},{C}], got {tuple(a.shape)}, {tuple(b.shape)}")
    dev = head.dev
    a = a.detach().to(device=dev, dtype=torch.float32).contiguous()
    b = b.detach().to(device=dev, dtype=torch.float32).contiguous()
    wh = None if img_wh is None else img_wh.to(device=dev, dtype=torch.float32).contiguous()
    out = dict(boxes=torch.empty(B, top_k, 4, device=dev), prob=torch.empty(B, top_k, device=dev),
               cls=torch.empty(B, top_k, dtype=torch.int32, device=dev),
               prior=torch.empty(B, top_k, dtype=torch.int32, device=dev),
               cnt=torch.empty(B, dtype=torch.int32, device=dev))
    with head._calls((_lib.WS_DETECT, B, int(max_candidates))) as (ws,):
        if from_scores:
            rc = head.lib.ssdhead_detect_from_scores(
                _ptr(a), _ptr(b), B, P, C, float(min_score), float(iou_thr), int(top_k), _ptr(wh), int(max_candidates),
                _ptr(out["boxes"]), _ptr(out["prob"]), _ptr(out["cls"]), _ptr(out["prior"]), _ptr(out["cnt"]),
                _ptr(ws), ws.numel(), _stream(dev))
        else:
            rc = head.lib.ssdhead_detect(
                _ptr(a), _ptr(b), _ptr(head.pri_cxcywh), B, P, C, float(min_score), float(iou_thr), int(top_k),
                _ptr(wh), int(max_candidates),
                _ptr(out["boxes"]), _ptr(out["prob"]), _ptr(out["cls"]), _ptr(out["prior"]), _ptr(out["cnt"]),
                _ptr(ws), ws.numel(), _stream(dev))
        _lib.check(rc, "ssdhead_detect")
    return out


def detect_fallbacks(head: MultiboxHead, B: int, max_candidates: int = 0) -> int:
    """Images of the LAST detect call with this batch size that the short-list route could not decide (they were served
    by the exhaustive kernels; the output is the same either way).  Synchronises the stream."""
    import ctypes
    n = ctypes.c_int32(-1)
    with head._calls((_lib.WS_DETECT, B, int(max_candidates))) as (ws,):
        _lib.check(head.lib.ssdhead_detect_fallbacks(_ptr(ws), ws.numel(), B, head.P, head.C, int(max_candidates),
                                                     ctypes.addressof(n), _stream(head.dev)), "ssdhead_detect_fallbacks")
    return int(n.value)


def detect(head: MultiboxHead, loc, conf, min_score=0.2, iou_thr=0.45, top_k=200, img_wh=None, max_candidates=0):
    return _detect(head, loc, conf, min_score, iou_thr, top_k, img_wh, max_candidates, False)


def detect_from_scores(head: MultiboxHead, boxes_cxcywh, probs, min_score=0.2, iou_thr=0.45, top_k=200,
                       img_wh=None, max_candidates=0):
    return _detect(head, boxes_cxcywh, probs, min_score, iou_thr, top_k, img_wh, max_candidates, True)


class _MultiboxLossLevelsFn(torch.autograd.Function):
    """``ssd()`` on per-level head tensors: inputs = L loc tensors then L conf tensors; the gradients come back per
    level in the same layout, so autograd continues straight into each conv (the permute is a view)."""

    @staticmethod
    def forward(ctx, head: MultiboxHead, gt: PackedGT, neg_ratio, pos_iou, L, need, *tensors):
        locs, confs = tensors[:L], tensors[L:]
        out = head.loss_levels(locs, confs, gt, with_grads=need, neg_ratio=neg_ratio, pos_iou=pos_iou)
        ctx.head = head
        ctx.meta = [(t.shape, t.device, t.dtype) for t in tensors]
        ctx.grads = (out["grad_loc"], out["grad_conf"]) if need else None
        a, b = out["losses"].unbind(0)
        return a, b

    @staticmethod
    def backward(ctx, g_loc_loss, g_conf_loss):
        if ctx.grads is None:
            raise RuntimeError("ssd_levels(): backward called twice (or without grad-requiring inputs)")
        gls, gcs = ctx.grads
        ctx.grads = None
        head = ctx.head
        gout = _upstream(head, g_loc_loss, g_conf_loss)
        for gl, gc in zip(gls, gcs):
            head.scale_grads(gl, gc, gout)
        outs = [g.reshape(shape).to(device=dev, dtype=dt) for g, (shape, dev, dt) in zip(list(gls) + list(gcs), ctx.meta)]
        return (None, None, None, None, None, None, *outs)


def multibox_loss_levels(head: MultiboxHead, loc_levels, conf_levels, gt_boxes, gt_classes,
                         neg_ratio: int = NEG_RATIO, pos_iou: float = POS_IOU):
    """(loc_loss, conf_loss) from per-level head tensors - ``ssd()`` without Model.py:212-235's permute/cat copies."""
    gt = PackedGT(gt_boxes, gt_classes, head.dev)
    L = len(conf_levels)
    need = torch.is_grad_enabled() and any(t.requires_grad for t in list(loc_levels) + list(conf_levels))
    return _MultiboxLossLevelsFn.apply(head, gt, neg_ratio, pos_iou, L, need, *loc_levels, *conf_levels)


def detect_levels(head: MultiboxHead, loc_levels, conf_levels, min_score=0.2, iou_thr=0.45, top_k=200, img_wh=None,
                  max_candidates=0):
    """``detect`` on per-level head tensors (same output dict)."""
    import ctypes
    st, locs, confs, B = head._levels(loc_levels, conf_levels)
    dev = head.dev
    wh = None if img_wh is None else img_wh.to(device=dev, dtype=torch.float32).contiguous()
    out = dict(boxes=torch.empty(B, top_k, 4, device=dev), prob=torch.empty(B, top_k, device=dev),
               cls=torch.empty(B, top_k, dtype=torch.int32, device=dev),
               prior=torch.empty(B, top_k, dtype=torch.int32, device=dev),
               cnt=torch.empty(B, dtype=torch.int32, device=dev))
    with head._calls((_lib.WS_DETECT, B, int(max_candidates))) as (ws,):
        _lib.check(head.lib.ssdhead_detect_levels(
            ctypes.addressof(st), _ptr(head.pri_cxcywh), B, head.P, head.C, float(min_score), float(iou_thr), int(top_k),
            _ptr(wh), int(max_candidates),
            _ptr(out["boxes"]), _ptr(out["prob"]), _ptr(out["cls"]), _ptr(out["prior"]), _ptr(out["cnt"]),
            _ptr(ws), ws.numel(), _stream(dev)), "ssdhead_detect_levels")
    return out



# ---------------------------------------------------------------------------------------------- CUDA graph capture
class _FixedWorkspaces(MultiboxHead):
    """A MultiboxHead whose workspaces are allocated and zero-filled by the first call that needs each of them, outside
    any capture, and then never resized, moved or re-zeroed: a captured graph keeps pointing at them, and the kernels
    leave every counter zeroed again.  Its callers keep the batch size and the gt capacity fixed, so each workspace has
    one size.  No events: an event recorded inside a capture cannot be waited on outside it, so the caller keeps its calls
    and replays on one stream."""

    _ordered = False

    def _workspace(self, which: int, B: int, n: int) -> torch.Tensor:
        cur = self._ws.get(which)
        if cur is None:
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("StaticHead: the first loss / loss_levels / detect call allocates and zero-fills its "
                                   "workspace and cannot be captured; make one eager call of it first (a warm-up step)")
            need = int(self.lib.ssdhead_workspace_bytes(which, B, self.P, self.C, n))
            if need == 0:
                raise RuntimeError(f"ssdhead: unsupported shape for this entry point (B={B}, P={self.P}, C={self.C})")
            with torch.cuda.device(self.dev):
                cur = torch.zeros(need, dtype=torch.uint8, device=self.dev)
            self._ws[which] = cur
        return cur


class _StaticGT:
    """Device gt buffers of fixed capacity in the ``pinned.gt_layout`` layout; ``sumG`` is the capacity (the kernels
    read the count from ``off[B]``)."""

    def __init__(self, B: int, capacity: int, dev: torch.device):
        from .pinned import gt_layout
        o0, o1, o2, total = gt_layout(capacity, B)
        self.B, self.sumG = B, capacity
        self.block = torch.zeros(total, dtype=torch.uint8, device=dev)
        self.boxes = self.block[o0:o0 + capacity * 16].view(torch.float32).view(capacity, 4)
        self.classes = self.block[o1:o1 + capacity * 4].view(torch.float32)
        self.off = self.block[o2:o2 + (B + 1) * 4].view(torch.int32)


class StaticHead:
    """The training-head step and detect of one fixed batch size, in a form that can be captured into a CUDA graph.

    It owns its device gt buffers (room for ``max_gt`` gts of ``batch`` images) and its workspaces, so a graph captured
    around ``loss`` / ``loss_levels`` (with ``backward()``) or ``detect`` stays valid: the kernels read the gt count
    from the offsets on the device.  Before each replay, ``load`` or ``load_packed`` writes the next batch's gts into
    the buffers, in stream order on the current stream; both refuse to run under capture.  The first call of
    ``loss`` / ``loss_levels`` / ``detect`` allocates its workspace and must be eager (a warm-up step).  One graph per
    object: two graphs of one object would share its gt buffers and workspaces.

        sh = StaticHead(priors, batch=32, max_gt=32 * 64, device="cuda")
        sh.load(boxes, classes); l, c = sh.loss(loc, conf); (l + c).backward()      # warm-up, eager
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            l, c = sh.loss(loc, conf); (l + c).backward()
        for boxes, classes in batches:
            sh.load(boxes, classes)            # or sh.load_packed(*collate.collate_gt(...))
            loc.copy_(...); conf.copy_(...); g.replay()
    """

    def __init__(self, priors: torch.Tensor, batch: int, max_gt: int, device=None, num_classes: int = 21):
        if torch.cuda.is_available() and torch.cuda.is_current_stream_capturing():
            raise RuntimeError("StaticHead: create it before capturing (it allocates its buffers)")
        self.B, self.max_gt = int(batch), int(max_gt)
        if self.B < 1 or self.max_gt < self.B:
            raise ValueError(f"StaticHead: batch must be >= 1 and max_gt >= batch (every image has a gt), got "
                             f"batch={batch}, max_gt={max_gt}")
        self.head = _FixedWorkspaces(priors, device, num_classes)
        self.dev = self.head.dev
        self.gt = _StaticGT(self.B, self.max_gt, self.dev)
        from .pinned import StagingPool
        self._pool = StagingPool()
        self._loaded = False

    # ------------------------------------------------------------------ gts, outside the graph
    def _refuse_capture(self, what: str) -> None:
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError(f"StaticHead.{what}() cannot be captured: call it before each replay, outside the graph")

    def _offsets(self, counts) -> np.ndarray:
        if len(counts) != self.B:
            raise ValueError(f"StaticHead holds {self.B} images, got {len(counts)}")
        bad = [i for i, n in enumerate(counts) if n <= 0]
        if bad:
            # the reference fails the same way on an image without objects (Losses.py:153, max over an empty dim)
            raise IndexError(f"image {bad[0]} has no ground-truth box: max() over an empty dimension")
        offs = np.zeros(self.B + 1, dtype=np.int32)
        np.cumsum(counts, out=offs[1:])
        if int(offs[-1]) > self.max_gt:
            raise ValueError(f"StaticHead: {int(offs[-1])} gts, more than max_gt = {self.max_gt}")
        return offs

    def _upload(self, st) -> None:
        """One copy of the whole staging block into the device buffers; the block returns to the pool behind an event."""
        cur = torch.cuda.current_stream(self.dev)
        self.gt.block.copy_(st.raw_t, non_blocking=True)
        if st.event is None:
            st.event = torch.cuda.Event()
        st.event.record(cur)
        self._pool.release(st, st.event)
        self._loaded = True

    def load(self, boxes: Sequence[torch.Tensor], classes: Sequence[torch.Tensor]) -> None:
        """Ragged gt lists (``ssd()``'s ``tr_bboxs`` / ``tr_classes``: B tensors of [n_i, 4] fractional xyxy and [n_i]
        class ids), on the host or on the device, into the device buffers."""
        self._refuse_capture("load")
        if len(classes) != len(boxes):
            raise ValueError(f"{len(boxes)} box lists but {len(classes)} class lists")
        offs = self._offsets([b.shape[0] if b.dim() > 0 else 0 for b in boxes])
        n = int(offs[-1])
        bx, cl = PackedGT._cat(boxes, 4), PackedGT._cat(classes, 0)
        if tuple(bx.shape) != (n, 4) or tuple(cl.shape) != (n,):
            raise ValueError(f"gt lists disagree: boxes {tuple(bx.shape)}, classes {tuple(cl.shape)}, {n} gts expected")
        if bx.device.type == "cpu" and cl.device.type == "cpu":
            st = self._pool.acquire(self.max_gt, self.B, exact=True)
            _staging_views(st)
            st.boxes_t[:n].copy_(bx)
            st.classes_t[:n].copy_(cl)
            st.offsets[:] = offs
            self._upload(st)
            return
        self.gt.boxes[:n].copy_(bx, non_blocking=True)
        self.gt.classes[:n].copy_(cl, non_blocking=True)
        self.gt.off.copy_(torch.from_numpy(offs).pin_memory(), non_blocking=True)
        self._loaded = True

    def load_packed(self, gt_xyxy, gt_cls, gt_off) -> None:
        """The packed layout of ``collate.collate_gt`` (boxes [n,4], classes [n], offsets int32 [B+1]): numpy arrays or
        tensors, on the host or on the device (device offsets are read back to check them: one synchronisation)."""
        self._refuse_capture("load_packed")
        off = gt_off.detach().cpu().numpy() if isinstance(gt_off, torch.Tensor) else np.asarray(gt_off)
        off = off.astype(np.int64).reshape(-1)
        if off.shape[0] != self.B + 1 or off[0] != 0:
            raise ValueError(f"StaticHead: expected {self.B + 1} offsets starting at 0, got {off.shape[0]}")
        offs = self._offsets(np.diff(off))
        n = int(offs[-1])
        if gt_xyxy.shape[0] < n or gt_cls.shape[0] < n:
            raise ValueError(f"StaticHead: the offsets list {n} gts, the arrays hold {gt_xyxy.shape[0]} boxes and "
                             f"{gt_cls.shape[0]} classes")
        if not any(isinstance(t, torch.Tensor) and t.is_cuda for t in (gt_xyxy, gt_cls)):
            st = self._pool.acquire(self.max_gt, self.B, exact=True)
            _staging_views(st)
            as_np = lambda a: a.detach().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
            st.boxes[:n] = as_np(gt_xyxy)[:n].reshape(n, 4)
            st.classes[:n] = as_np(gt_cls)[:n].reshape(n)
            st.offsets[:] = offs
            self._upload(st)
            return
        as_t = lambda a: a if isinstance(a, torch.Tensor) else torch.from_numpy(np.asarray(a))
        self.gt.boxes[:n].copy_(as_t(gt_xyxy)[:n].reshape(n, 4), non_blocking=True)
        self.gt.classes[:n].copy_(as_t(gt_cls)[:n].reshape(n), non_blocking=True)
        self.gt.off.copy_(torch.from_numpy(offs).pin_memory(), non_blocking=True)
        self._loaded = True

    # ------------------------------------------------------------------ capturable calls
    def _require_loaded(self) -> None:
        if not self._loaded:
            raise RuntimeError("StaticHead: load() or load_packed() the gts before the first loss call")

    def loss(self, loc: torch.Tensor, conf: torch.Tensor, neg_ratio: int = NEG_RATIO, pos_iou: float = POS_IOU):
        """(loc_loss, conf_loss) as 0-dim tensors with grad_fn, as ``ssd()`` returns them, on the loaded gts."""
        self._require_loaded()
        need = torch.is_grad_enabled() and (loc.requires_grad or conf.requires_grad)
        return _MultiboxLossFn.apply(loc, conf, self.head, self.gt, neg_ratio, pos_iou, None, need)

    def loss_levels(self, loc_levels, conf_levels, neg_ratio: int = NEG_RATIO, pos_iou: float = POS_IOU):
        """``loss`` on per-level head tensors, as ``ssd_levels()``."""
        self._require_loaded()
        L = len(conf_levels)
        need = torch.is_grad_enabled() and any(t.requires_grad for t in list(loc_levels) + list(conf_levels))
        return _MultiboxLossLevelsFn.apply(self.head, self.gt, neg_ratio, pos_iou, L, need, *loc_levels, *conf_levels)

    def detect(self, loc: torch.Tensor, conf: torch.Tensor, min_score: float = 0.2, iou_thr: float = 0.45,
               top_k: int = 200, img_wh: Optional[torch.Tensor] = None):
        """The ``inference_batch`` dict (boxes, prob, cls, prior, cnt).  ``img_wh`` [B,2], if given, must already be on
        this device: a host copy cannot be captured."""
        if int(loc.shape[0]) != self.B:
            raise ValueError(f"StaticHead holds {self.B} images, got a batch of {int(loc.shape[0])}")
        if img_wh is not None and (not isinstance(img_wh, torch.Tensor) or img_wh.device != self.dev):
            raise ValueError(f"StaticHead.detect: img_wh must be a tensor on {self.dev} (a host copy cannot be captured)")
        return _detect(self.head, loc, conf, min_score, iou_thr, top_k, img_wh, 0, False)
