"""Drop-in for the hot-path functions of the reference's ``Util.py`` (same names, argument meaning
and return types), backed by the sm_100a kernels of libssdhead.so.

Mirrored (reference file:line):
  create_priors_ssd300   Util.py:105-137   prior table (host, float64 -> float32, bit-identical)
  xywh_to_xyxy           Util.py:93-96     | xyxy_to_xywh        Util.py:57-63 (returns a CPU tensor)
  gcxgcy_to_cxcy         Util.py:86-91     | get_offsets_coords  Util.py:98-102
  find_intersection      Util.py:252-265   | get_jaccard_tensor1 Util.py:288-301
  get_jaccard_tensor11   Util.py:303-316   (CPU ONLY on purpose: it runs inside DataLoader workers)
  map_prior_to_bb        Util.py:333-352   | subsampling         Util.py:555-560 (used by Model.py)
  class_to_label / label_to_class  Util.py:26-31 | device  Util.py:12-13

Like the reference, the functions move host inputs to ``device`` (CUDA when available) and return
tensors there; inputs already on a CUDA device are computed on, and returned on, that device (the kernels run
there whatever the current device is).  There is no CPU fallback for them: without a CUDA device they raise.  The one exception
is ``get_jaccard_tensor11`` (and ``find_intersection`` when it is handed CPU tensors by it), which the
reference keeps off the GPU deliberately because forked DataLoader workers must not touch CUDA
(Util.py:305, Util.py:697).

Names of the reference's ``Util`` that are NOT on the head path (dataset lists, augmentation ``transform``,
drawing, ``get_map``) are resolved lazily from the reference's own module if it is importable as
``Util_reference`` or found through ``SSD_REFERENCE_DIR``; importing this module never parses the VOC
annotation set or needs matplotlib (SURVEY.md section 3.3).
"""
from __future__ import annotations

import importlib
import importlib.util
import os
import sys

import numpy as np
import torch

from . import _lib
from .priors import make_priors, SSD300_SPEC

use_cuda = torch.cuda.is_available()
device = torch.device("cuda" if use_cuda else "cpu")

class_to_label = ['aeroplane', 'bicycle', 'bird', 'boat', 'bottle', 'bus', 'car', 'cat', 'chair', 'cow', 'diningtable',
                  'dog', 'horse', 'motorbike', 'person', 'pottedplant', 'sheep', 'sofa', 'train', 'tvmonitor', "bg"]
label_to_class = {name: idx for idx, name in enumerate(class_to_label)}


def _cuda_device(*inputs) -> torch.device:
    """The device of the first CUDA tensor among ``inputs``, else ``device``."""
    if not torch.cuda.is_available():
        raise RuntimeError("objectdetection_ssd_b200.Util: no CUDA device - these functions have no CPU fallback")
    for t in inputs:
        if isinstance(t, torch.Tensor) and t.is_cuda:
            return t.device
    d = torch.device(device)
    if d.type != "cuda":
        d = torch.device("cuda")
    return torch.device("cuda", torch.cuda.current_device() if d.index is None else d.index)


def _f32(t, dev):
    return torch.as_tensor(t).detach().to(device=dev, dtype=torch.float32).contiguous()


def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream


def create_priors_ssd300():
    """8732 x 4 (cx, cy, w, h) float32, clamped to [0, 1] (Util.py:105-137)."""
    print("-----------------------create priors-------------------")
    return make_priors(SSD300_SPEC)


def _box_op(name, a, b=None):
    dev = _cuda_device(a, b)
    a = _f32(a, dev).reshape(-1, 4)
    out = torch.empty_like(a)
    lib = _lib.load()
    with torch.cuda.device(dev):
        if b is None:
            rc = getattr(lib, name)(a.data_ptr(), out.data_ptr(), a.shape[0], _stream(dev))
        else:
            b = _f32(b, dev).reshape(-1, 4)
            if b.shape[0] != a.shape[0]:
                raise RuntimeError(f"The size of tensor a ({a.shape[0]}) must match the size of tensor b ({b.shape[0]})")
            rc = getattr(lib, name)(a.data_ptr(), b.data_ptr(), out.data_ptr(), a.shape[0], _stream(dev))
    _lib.check(rc, name)
    return out


class _BoxOpFn(torch.autograd.Function):
    """The reference's box functions are plain torch expressions and therefore differentiable; the kernels are not
    seen by autograd, so when an input requires grad the (elementwise, closed-form) backward is supplied here.  It is
    off the hot path: the loss kernels produce their own gradients."""

    @staticmethod
    def forward(ctx, name, a, b):
        out = _box_op(name, a, b)
        ctx.name = name
        ctx.save_for_backward(a.detach(), b.detach() if b is not None else None, out)
        return out

    @staticmethod
    def backward(ctx, g):
        a, b, out = ctx.saved_tensors
        dev = out.device
        g = g.to(dev)
        ga = gb = None
        if ctx.name == "ssdhead_cxcywh_to_xyxy":            # [c - wh/2, c + wh/2]
            ga = torch.cat([g[:, :2] + g[:, 2:], (g[:, 2:] - g[:, :2]) / 2], 1)
        elif ctx.name == "ssdhead_decode":                    # [g_c * p_wh / 10 + p_c, exp(g_wh / 5) * p_wh]
            pb = b.to(dev).reshape(-1, 4)
            ga = torch.cat([g[:, :2] * pb[:, 2:] / 10, g[:, 2:] * out[:, 2:] / 5], 1)
            if ctx.needs_input_grad[2]:
                aa = a.to(dev).reshape(-1, 4)
                gb = torch.cat([g[:, :2], g[:, :2] * aa[:, :2] / 10 + g[:, 2:] * out[:, 2:] / pb[:, 2:]], 1)
        elif ctx.name == "ssdhead_encode":                    # [(c - p_c) / (p_wh / 10), log(wh / p_wh) * 5]
            aa, pb = a.to(dev).reshape(-1, 4), b.to(dev).reshape(-1, 4)
            ga = torch.cat([g[:, :2] * 10 / pb[:, 2:], g[:, 2:] * 5 / aa[:, 2:]], 1)
            if ctx.needs_input_grad[2]:
                gb = torch.cat([-g[:, :2] * 10 / pb[:, 2:], -g[:, :2] * out[:, :2] / pb[:, 2:] - g[:, 2:] * 5 / pb[:, 2:]], 1)
        if ga is not None:
            ga = ga.reshape(a.shape).to(a.device)
        if gb is not None:
            gb = gb.reshape(b.shape).to(b.device)
        return None, ga, gb


def _box_fn(name, a, b=None):
    ts = [t for t in (a, b) if isinstance(t, torch.Tensor)]
    if torch.is_grad_enabled() and any(t.requires_grad for t in ts):
        return _BoxOpFn.apply(name, torch.as_tensor(a), None if b is None else torch.as_tensor(b))
    return _box_op(name, a, b)


def xywh_to_xyxy(box):
    return _box_fn("ssdhead_cxcywh_to_xyxy", box)


def xyxy_to_xywh(anchors):
    # the reference goes through numpy and hands back a CPU tensor (Util.py:58-63): not differentiable there either
    return _box_op("ssdhead_xyxy_to_cxcywh", anchors).cpu()


def gcxgcy_to_cxcy(gcxgcy, priors_cxcy):
    return _box_fn("ssdhead_decode", gcxgcy, priors_cxcy)


def get_offsets_coords(cxcy, priors_cxcy):
    return _box_fn("ssdhead_encode", cxcy, priors_cxcy)


def _pair_matrix(name, set_1, set_2):
    dev = _cuda_device(set_1, set_2)
    a, b = _f32(set_1, dev).reshape(-1, 4), _f32(set_2, dev).reshape(-1, 4)
    out = torch.empty(a.shape[0], b.shape[0], dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(getattr(_lib.load(), name)(a.data_ptr(), a.shape[0], b.data_ptr(), b.shape[0], out.data_ptr(),
                                              _stream(dev)), name)
    return out


def _intersection_cpu(set_1, set_2):
    lo = torch.max(set_1[:, :2].unsqueeze(1), set_2[:, :2].unsqueeze(0))
    hi = torch.min(set_1[:, 2:].unsqueeze(1), set_2[:, 2:].unsqueeze(0))
    d = torch.clamp(hi - lo, min=0)
    return d[:, :, 0] * d[:, :, 1]


def find_intersection(set_1, set_2):
    """[n1, n2] intersection areas of corner-form boxes (Util.py:252-265).  CPU tensors stay on the CPU
    (the augmentation path of the DataLoader workers); CUDA tensors use the kernel."""
    if not set_1.is_cuda and not set_2.is_cuda:
        return _intersection_cpu(set_1, set_2)
    return _pair_matrix("ssdhead_intersection_matrix", set_1, set_2)


def get_jaccard_tensor1(box1_xyxy, box2_xyxy):
    """[n1, n2] IoU on ``device`` (Util.py:288-301)."""
    return _pair_matrix("ssdhead_iou_matrix", box1_xyxy, box2_xyxy)


def get_jaccard_tensor11(box1_xyxy, box2_xyxy):
    """CPU-only IoU used by the augmentation inside DataLoader workers (Util.py:303-316, caller Util.py:697)."""
    inter = _intersection_cpu(box1_xyxy, box2_xyxy)
    a1 = (box1_xyxy[:, 2] - box1_xyxy[:, 0]) * (box1_xyxy[:, 3] - box1_xyxy[:, 1])
    a2 = (box2_xyxy[:, 2] - box2_xyxy[:, 0]) * (box2_xyxy[:, 3] - box2_xyxy[:, 1])
    return inter / (a1.unsqueeze(1) + a2.unsqueeze(0) - inter)


def map_prior_to_bb(jacc, classes, threshold=0.5):
    """Single-image match from a jaccard matrix [n_objects, n_priors] (Util.py:333-352).
    Returns (class_forEach_prior float [P] with 20 = background, obj_forEach_prior int64 [P])."""
    dev = _cuda_device(jacc, classes)
    j = _f32(jacc, dev)
    if j.dim() != 2 or j.shape[0] == 0:
        raise IndexError("max(): Expected reduction dim 0 to have non-zero size.")
    G, P = int(j.shape[0]), int(j.shape[1])
    cl = _f32(classes, dev).reshape(-1)
    cls = torch.empty(P, dtype=torch.float32, device=dev)
    obj = torch.empty(P, dtype=torch.int64, device=dev)
    ov = torch.empty(P, dtype=torch.float32, device=dev)
    bp = torch.empty(G, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().ssdhead_match_from_iou(j.data_ptr(), cl.data_ptr(), G, P, float(threshold), 20,
                                                      cls.data_ptr(), obj.data_ptr(), ov.data_ptr(), bp.data_ptr(),
                                                      _stream(dev)), "ssdhead_match_from_iou")
    return cls.to(dtype=torch.as_tensor(classes).dtype), obj      # classes[obj] keeps the dtype of `classes`


def get_map(det_boxes, det_classes, det_scores, gt_boxes, gt_classes):
    """VOC 11-point interpolated average precision per class (Util.py:783-885), on the GPU.

    Arguments as in the reference: per-image lists of tensors (detections: boxes [n,4], classes [n], scores [n];
    ground truth: boxes [m,4], classes [m]).  Returns ``{class_id: AP}`` for the 20 foreground classes (numpy
    float64).  Equal scores rank by the lower detection index (the reference's sort leaves ties open)."""
    dev = _cuda_device(*(x for lists in (det_boxes, det_scores, gt_boxes) for x in lists[:1]))
    n_img = len(det_boxes)
    if n_img == 0 or len(gt_boxes) != n_img:
        raise ValueError("get_map: detections and ground truth must be per-image lists of the same, non-zero length")

    def pack(lists, width, dtype):
        parts = [torch.as_tensor(x).reshape(-1, width) if width else torch.as_tensor(x).reshape(-1) for x in lists]
        off = [0]
        for p_ in parts:
            off.append(off[-1] + int(p_.shape[0]))
        shape = (0, width) if width else (0,)
        cat = torch.cat(parts) if off[-1] else torch.zeros(shape)
        return cat.to(device=dev, dtype=dtype).contiguous(), off

    db, doff = pack(det_boxes, 4, torch.float32)
    dc, _ = pack(det_classes, 0, torch.int32)
    ds, _ = pack(det_scores, 0, torch.float32)
    gb, goff = pack(gt_boxes, 4, torch.float32)
    gc, _ = pack(gt_classes, 0, torch.float32)
    N, M = doff[-1], goff[-1]
    d_off = torch.tensor(doff, dtype=torch.int32, device=dev)
    g_off = torch.tensor(goff, dtype=torch.int32, device=dev)
    levels = torch.arange(0, 1.1, 0.1).to(device=dev, dtype=torch.float64)      # the float32 values of Util.py:875
    ap = torch.zeros(20, dtype=torch.float64, device=dev)
    lib = _lib.load()
    ws = torch.empty(int(lib.ssdhead_voc_ap_workspace_bytes(N, M, 20)), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ssdhead_voc_ap(db.data_ptr() if N else None, dc.data_ptr() if N else None,
                                      ds.data_ptr() if N else None, d_off.data_ptr(), N, gb.data_ptr() if M else None,
                                      gc.data_ptr() if M else None, g_off.data_ptr(), M, n_img, 20, 0.5, levels.data_ptr(),
                                      ap.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev)), "ssdhead_voc_ap")
    out = ap.cpu().numpy()
    return {c: out[c] for c in range(20)}


def get_img_sz(img_path):
    """(width, height) of an image file (Util.py:226-228).  Local, so ``inference(..., toDraw=False)`` needs nothing of
    the reference's dataset side beyond the path itself."""
    from PIL import Image
    with Image.open(img_path) as im:
        return im.size


def subsampling(x, step):
    """Strided sub-sampling used by Model.py for the fc6/fc7 surgery (Util.py:555-560); plain indexing."""
    for d, s in enumerate(step):
        if s is None:
            continue
        x = x.index_select(dim=d, index=torch.arange(start=0, end=x.shape[d], step=s).long().to(x.device))
    return x


# ------------------------------------------------------------------------------------------------------------
# everything else of the reference's Util (dataset lists, augmentation, drawing, get_map) is out of the head path:
# forwarded lazily to the reference's own module when it can be found, never imported eagerly.
_reference_util = None


def _load_reference_util():
    global _reference_util
    if _reference_util is not None:
        return _reference_util
    for name in ("Util_reference",):
        try:
            _reference_util = importlib.import_module(name)
            return _reference_util
        except ImportError:
            pass
    ref_dir = os.environ.get("SSD_REFERENCE_DIR")
    if ref_dir and os.path.isfile(os.path.join(ref_dir, "Util.py")):
        spec = importlib.util.spec_from_file_location("Util_reference", os.path.join(ref_dir, "Util.py"))
        mod = importlib.util.module_from_spec(spec)
        sys.path.insert(0, ref_dir)
        try:
            spec.loader.exec_module(mod)
        finally:
            sys.path.remove(ref_dir)
        sys.modules["Util_reference"] = mod
        _reference_util = mod
        return mod
    return None


def __getattr__(name):
    mod = _load_reference_util()
    if mod is not None and hasattr(mod, name):
        return getattr(mod, name)
    raise AttributeError(
        f"objectdetection_ssd_b200.Util has no attribute {name!r}: only the SSD head path is implemented here; "
        "set SSD_REFERENCE_DIR (or provide a module named Util_reference) to forward dataset / augmentation / "
        "drawing names to the reference's own Util.py")
