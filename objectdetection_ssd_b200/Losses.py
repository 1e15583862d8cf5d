"""Drop-in for the reference's ``Losses.py`` call surface (same names, arguments and returns), backed by
the sm_100a kernels of libssdhead.so through the C ABI (include/ssdhead.h).

  ssd(outputs, tr_classes, tr_bboxs) -> (loc_loss, conf_loss)            Losses.py:119-134
  ssd1_(loc, conf, tr_bbox, tr_class, jaccard, indices) -> (c_loss, loc_loss)   Losses.py:136-199
  ssd_old(outputs, tr_classes, tr_bboxs) / ssd1(loc, conf, tr_bbox, tr_class)   Losses.py:100-117, 201-225
  inference(l_, c_, index, top_k, phase, toDraw, min_score, iou_threshold)      Losses.py:11-98
  ancs_xywh, ancs_xyxy, device                                           Losses.py:6-9
  obj_forEach_prior___  (debug tap: class per prior of the last ssd() call)     Losses.py:172-173

``train_function.py`` can keep ``from Losses import *`` (see INTEGRATION.md / ``dropin/``): ``ssd`` returns two
0-dim tensors with ``grad_fn``; ``(loss1 + loss2).backward()`` delivers the dense gradients the fused kernels
wrote during the forward call.  Semantics reproduced on purpose: background is class 20, the loc loss is plain
L1 (mean over 4*Npos), normalisation is by the batch-global positive count, top_k is a global post-NMS cap,
boxes are not clamped.  An image without ground truth raises IndexError, as the reference does.
"""
from __future__ import annotations

import torch

from . import Util as _U
from .Util import (class_to_label, label_to_class, create_priors_ssd300, xywh_to_xyxy, xyxy_to_xywh,       # noqa: F401
                   gcxgcy_to_cxcy, get_offsets_coords, find_intersection, get_jaccard_tensor1,
                   get_jaccard_tensor11, map_prior_to_bb, subsampling)
from .head import (MultiboxHead, PackedGT, StaticHead, multibox_loss, detect as _detect, multibox_loss_levels,  # noqa: F401
                   detect_levels as _detect_levels, refuse_capture as _refuse_capture)
from .priors import cxcywh_to_xyxy_host

ancs_xywh = create_priors_ssd300()
ancs_xyxy = cxcywh_to_xyxy_host(ancs_xywh)          # same fp32 ops as xywh_to_xyxy, kept on the CPU like the reference
use_cuda = torch.cuda.is_available()
device = torch.device("cuda" if use_cuda else "cpu")

process_group = None        # set to a torch.distributed group when the batch is sharded by image over several GPUs

_heads = {}
_last = {}


def _head(dev=None) -> MultiboxHead:
    """MultiboxHead for the current module-global prior table (the reference reads ``ancs_xywh`` at call time,
    Losses.py:23,129,181, so overwriting it - e.g. with a 24 564-prior table - must take effect)."""
    if dev is None:
        dev = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else None
    key = (str(dev), id(ancs_xywh), tuple(ancs_xywh.shape))
    h = _heads.get(key)
    if h is None:
        _heads.clear()
        h = MultiboxHead(ancs_xywh, dev if dev is not None else "cuda")
        _heads[key] = h
    return h


def _dev_of(t):
    return t.device if (isinstance(t, torch.Tensor) and t.is_cuda) else None


def ssd(outputs, tr_classes, tr_bboxs):
    """Batch multibox loss.  ``outputs`` = (loc [B,P,4], conf [B,P,21]); ``tr_classes`` / ``tr_bboxs`` = lists of
    B tensors ([n_i] class ids, [n_i,4] fractional xyxy).  Returns (loc_loss, conf_loss).  Not capturable into a CUDA
    graph (it raises under capture): ``StaticHead`` is."""
    _refuse_capture("ssd()")
    loc, conf = outputs
    head = _head(_dev_of(loc))
    _last.clear()
    _last.update(head=head, boxes=tr_bboxs, classes=tr_classes)     # for the obj_forEach_prior___ tap, built on demand
    return multibox_loss(head, loc, conf, tr_bboxs, tr_classes, group=process_group)


def ssd1_(pred_bb_offset, pred_class_score, tr_bbox, tr_class, jaccard=None, indices=None):
    """The reference's inner function: same computation, returns (c_loss, loc_loss) - swapped w.r.t. ``ssd``
    (Losses.py:199).  ``jaccard`` / ``indices`` are accepted for signature compatibility; the IoU of the gt
    boxes against the module's prior table is recomputed inside the match kernel, bit-identically."""
    lb, lc = ssd((pred_bb_offset, pred_class_score), tr_class, tr_bbox)
    return lc, lb


def ssd1(pred_bb_offset, pred_class_score, tr_bbox, tr_class):
    """Single-image loss with per-image normalisation (Losses.py:201-225).  Returns (c_loss, loc_loss)."""
    lb, lc = ssd((pred_bb_offset.unsqueeze(0), pred_class_score.unsqueeze(0)), [tr_class], [tr_bbox])
    return lc, lb


def ssd_old(outputs, tr_classes, tr_bboxs):
    """Legacy variant: mean over the batch of per-image losses (Losses.py:100-117).  Returns (loc, conf)."""
    loc, conf = outputs
    bs = len(tr_bboxs)
    lbb = 0.0
    lc = 0.0
    for l, c, b, k in zip(loc, conf, tr_bboxs, tr_classes):
        lc_, lbb_ = ssd1(l, c, b, k)
        lbb = lbb + lbb_
        lc = lc + lc_
    return lbb / bs, lc / bs


def head_levels(loc_maps, conf_maps, num_classes=21):
    """The twelve conv outputs of the head (``Model.py:212-233``: per level a loc map [B, A*4, H, W] and a conf map
    [B, A*21, H, W]) as per-level row tensors [B, H*W*A, 4] / [B, H*W*A, 21].  ``permute(0, 2, 3, 1)`` is what the
    reference does; for a channels_last (NHWC) conv output it is a pure view, so neither the ``.contiguous()`` copy nor
    the ``torch.cat`` of Model.py:234-235 ever happens."""
    locs = [m.permute(0, 2, 3, 1).reshape(m.shape[0], -1, 4) for m in loc_maps]
    confs = [m.permute(0, 2, 3, 1).reshape(m.shape[0], -1, num_classes) for m in conf_maps]
    return locs, confs


def ssd_levels(outputs, tr_classes, tr_bboxs):
    """``ssd`` on per-level head tensors (SURVEY.md 8(f) #3): ``outputs`` = (list of loc [B, n_l, 4], list of conf
    [B, n_l, 21]) - e.g. from ``head_levels`` - in the prior order of ``create_priors_ssd300``.  Same value and
    gradients as ``ssd(torch.cat(...))``, bit for bit, without ever building the concatenated tensors."""
    _refuse_capture("ssd_levels()")
    locs, confs = outputs
    head = _head(_dev_of(confs[0]))
    _last.clear()
    _last.update(head=head, boxes=tr_bboxs, classes=tr_classes)
    return multibox_loss_levels(head, list(locs), list(confs), tr_bboxs, tr_classes)


def inference_batch_levels(loc_levels, conf_levels, top_k=200, min_score=0.2, iou_threshold=0.45, img_wh=None,
                           max_candidates=0):
    """``inference_batch`` on per-level head tensors."""
    _refuse_capture("inference_batch_levels()")
    return _detect_levels(_head(_dev_of(conf_levels[0])), list(loc_levels), list(conf_levels), min_score, iou_threshold,
                          top_k, img_wh, max_candidates)


def inference_batch(loc, conf, top_k=200, min_score=0.2, iou_threshold=0.45, img_wh=None, max_candidates=0):
    """Batched detect front end (SURVEY.md 8(f) #2): loc [B,P,4], conf [B,P,21] -> dict of padded
    [B,top_k,...] tensors + counts; ``img_wh`` [B,2] scales the boxes to pixels (Losses.py:87-89).  Under CUDA graph
    capture use ``StaticHead.detect``."""
    _refuse_capture("inference_batch()")
    return _detect(_head(_dev_of(loc)), loc, conf, min_score, iou_threshold, top_k, img_wh, max_candidates)


def _image_size(phase, index):
    """(w, h) by which ``inference`` scales its boxes (Losses.py:87-89).  The reference looks the file up through the
    dataset lists, ``get_img_sz(all_images[phase][index])``; that still works when those lists are available (they are
    the out-of-scope dataset side, forwarded from the reference's own Util).  So that the drop-in also works WITHOUT
    them, ``index`` may be the image path itself or a ``(w, h)`` pair."""
    if isinstance(index, (tuple, list)) and len(index) == 2:
        return float(index[0]), float(index[1])
    if isinstance(index, (str, bytes)) or hasattr(index, "__fspath__"):
        return _U.get_img_sz(index)
    return _U.get_img_sz(_U.all_images[phase][index])


def inference(l_, c_, index, top_k=200, phase='train', toDraw=True, min_score=0.2, iou_threshold=0.45):
    """Single-image detect.  ``l_`` [P,4] predicted offsets, ``c_`` [P,21] logits.  Returns
    (pred_bboxes [K,4] pixel xyxy, classes int64 [K], probs [K]) with K <= top_k, or ([], [], []) when
    nothing passes ``min_score`` (Losses.py:62-63)."""
    _refuse_capture("inference()")
    w, h = _image_size(phase, index)
    out = _detect(_head(_dev_of(l_)), l_.unsqueeze(0), c_.unsqueeze(0), min_score, iou_threshold, top_k,
                  torch.tensor([[float(w), float(h)]]), 0)
    k = int(out["cnt"][0])            # one host sync per image (the reference has 20, Losses.py:33)
    if k == 0:
        return [], [], []
    boxes, cls, prob = out["boxes"][0, :k], out["cls"][0, :k].long(), out["prob"][0, :k]
    if toDraw:
        labels = [class_to_label[i] for i in cls.tolist()]
        _U.draw_image_with_ancs_xyxy(_U.all_images[phase][index], boxes, labels, prob)
    return boxes, cls, prob


def __getattr__(name):
    if name == "obj_forEach_prior___":
        # the reference leaves the class-per-prior map of the last call in this global (Losses.py:172-173);
        # here it is produced on demand so the hot path does not pay for a debug tap
        if not _last:
            raise AttributeError("obj_forEach_prior___ is only defined after a call to ssd()")
        head = _last["head"]
        m = head.match(PackedGT([b.detach() for b in _last["boxes"]], [c.detach() for c in _last["classes"]], head.dev),
                       want_maps=True)
        return m["cls"].to(torch.float32)
    return getattr(_U, name)
