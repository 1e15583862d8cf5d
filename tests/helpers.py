"""Shared input builders for the parity tests (seeded, identical bits for oracle and kernels)."""
import numpy as np
import torch

from objectdetection_ssd_b200 import synth
from oracle import ssd_oracle as O


def priors(kind="ssd300"):
    if kind == "ssd300":
        return O.make_priors()
    if kind == "ssd512":
        return O.make_priors(**O.SSD512)
    raise ValueError(kind)


def train_inputs(seed, B, P, min_gt=1, max_gt=10, C=21):
    gb, gc = synth.make_gt(seed, B, min_gt, max_gt)
    loc, conf = synth.make_head(seed, B, P, C)
    tb = [torch.from_numpy(b) for b in gb]
    tc = [torch.from_numpy(c) for c in gc]
    return torch.from_numpy(loc), torch.from_numpy(conf), tb, tc


def detect_inputs(seed, B, P, bg_bias=6.0, C=21):
    loc, conf = synth.make_head(seed, B, P, C, loc_scale=0.5, bg_bias=bg_bias)
    return torch.from_numpy(loc), torch.from_numpy(conf)


def unpack_mask(mask_i32: torch.Tensor, P: int) -> torch.Tensor:
    """uint32 bit mask [B, ceil(P/32)] (stored as int32) -> bool [B,P]."""
    m = mask_i32.cpu().numpy().view(np.uint32)
    bits = ((m[:, :, None] >> np.arange(32, dtype=np.uint32)[None, None, :]) & 1).astype(bool)
    return torch.from_numpy(bits.reshape(m.shape[0], -1)[:, :P])


# ---------------------------------------------------------------------------------------------------------------
# Boundary proof for the FUSED detect path (own softmax / decode on the device).  CUDA's ex2.approx / expf and ATen's
# exp differ in the last bits, so a detection may differ from the oracle's - but only for a reason:
#   (a) its OWN probability is within its error bound of `min_score` (the candidate itself flips; it ranks last in its
#       class, so nothing else can change because of it);
#   (b) its class holds a pair (box kept by either side, candidate) whose IoU is within IOU_REL of the NMS threshold (a
#       suppression flips, and the greedy sweep of THAT class may cascade);
#   (c) its class holds a pair (box kept by either side, overlapping candidate: IoU >= the threshold, within IOU_REL)
#       whose probabilities are within their two error bounds of each other (their sweep order may flip - e.g. two
#       candidates at 1.0 in fp32 where one side rounds a probability 1 - 1e-8 to 1.0 and the other to the float below -
#       and with it which of the two suppresses the other; the class's sweep may cascade);
#   (d) more than top_k survive and it sits at the global cut: its probability is within the two error bounds of the
#       k-th largest, or it is at / below the cut while some class has a (b) or (c) event (one more or one fewer box
#       kept above moves the cut).
# A difference without such an event is a genuine error.  The error bounds are per candidate (softmax_f64 and
# decode_f64 below); decoded boxes differ by a few ulp (expf), their IoU by < 1e-5 relative.
EPS = 2.0 ** -23                 # one ulp of fp32 relative to the value, at most
IOU_REL = 1e-5


def softmax_f64(conf_i):
    """float64 softmax of fp32 logits [..., C] and a bound on |fp32 softmax - float64 softmax| per entry.

    Derived the way the CE bound of test_gpu_trained_regime.py is.  The kernel computes d_q = x_q - max, e_q =
    ex2.approx(d_q log2 e) with a relative error <= (2 + 1.16 |d_q|) ulp (csrc/common.cuh), s = sum_q e_q, inv = 1 / s and
    p_q = e_q * inv.  Per term: (2 + 2 |d_q|) eps (the ex2 error plus the |d_q| / 2 ulp of rounding d_q).  The C - 1
    additions round by half an ulp of a partial sum <= s each, so s is off by eps ((C - 1) / 2 + X) relative, X =
    sum_q (2 + 2 |d_q|) e_q / s; 1 / s and the product round once each.  So
        |p_q - p64_q| <= p64_q eps (3 + 2 |d_q| + (C - 1) / 2 + X)  +  2^-125,
    the absolute part for terms below 2^-126 that ex2.approx.ftz flushes.  ATen's fp32 softmax (1-ulp exp, another
    summation order, a division) stays inside the same bound.  Second-order terms are covered by a factor 1.001."""
    x = np.asarray(conf_i, np.float64)
    C = x.shape[-1]
    with np.errstate(invalid="ignore", over="ignore"):
        d = x - x.max(-1, keepdims=True)
        e = np.exp(d)
        s = e.sum(-1, keepdims=True)
        p = e / s
        X = ((2.0 + 2.0 * np.abs(d)) * e).sum(-1, keepdims=True) / s
        bound = 1.001 * p * EPS * (3.0 + 2.0 * np.abs(d) + (C - 1) / 2.0 + X) + 2.0 ** -125
    return p, bound


def decode_f64(loc_i, pri):
    """float64 decode + corner form of fp32 offsets [P,4] on priors [P,4] (Util.py:86-96) and a bound per coordinate.

    fp32 computes cx = g_x pw / 10 + px (three roundings: |g_x pw / 10| eps + |cx| eps / 2) and w = exp(g_w / 5) pw
    (g_w / 5 rounds: |g_w| / 10 eps relative through exp; expf <= 2 ulp; the product eps / 2), then x1 = cx - w / 2
    (w / 2 is exact; one more rounding of |x1| eps / 2).  Returns (xyxy float64 [P,4], bound [P,4])."""
    g = np.asarray(loc_i, np.float64)
    pr = np.asarray(pri, np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        c = g[:, :2] * pr[:, 2:] / 10.0 + pr[:, :2]
        wh = np.exp(g[:, 2:] / 5.0) * pr[:, 2:]
        xyxy = np.concatenate([c - wh / 2.0, c + wh / 2.0], 1)
        ec = np.abs(g[:, :2] * pr[:, 2:] / 10.0) * EPS + np.abs(c) * EPS / 2.0
        ew = wh * EPS * (np.abs(g[:, 2:]) / 10.0 + 2.5)
        bound = 1.001 * (np.concatenate([ec, ec], 1) + np.concatenate([ew, ew], 1) / 2.0 + np.abs(xyxy) * EPS / 2.0) + 2.0 ** -140
    return xyxy, bound


def explain_detect_mismatches(loc_i, conf_i, pri, min_score, iou_thr, top_k, ours, ref):
    """``ours`` / ``ref``: sets of (class, prior) detections of one image.  Returns (n_mismatches, unexplained list)."""
    import torch.nn.functional as F
    diff = (ours - ref) | (ref - ours)
    if not diff:
        return 0, []
    probs = F.softmax(conf_i, dim=1)
    p64, pb = softmax_f64(conf_i.numpy())
    boxes = O.cxcywh_to_xyxy(O.decode(loc_i, pri))
    fragile = set()                                             # classes with a (b) or (c) event
    for c in {c for c, _ in diff}:
        # only a box that one of the two sides KEPT can suppress anything: pairs (kept box, any candidate of the class)
        cand = torch.from_numpy(np.nonzero(p64[:, c] + pb[:, c] >= min_score)[0])
        kept = torch.tensor(sorted({p for cc, p in (ours | ref) if cc == c}), dtype=torch.long)
        if cand.numel() > 0 and kept.numel() > 0:
            iou = O.iou_matrix(boxes[kept], boxes[cand])
            iou[kept[:, None] == cand[None, :]] = 0
            near_thr = (iou - iou_thr).abs() <= IOU_REL * iou_thr                                  # (b)
            ki, ci = kept.numpy(), cand.numpy()
            close = np.abs(p64[ki, c][:, None] - p64[ci, c][None, :]) <= pb[ki, c][:, None] + pb[ci, c][None, :]
            order = (iou >= iou_thr * (1 - IOU_REL)) & torch.from_numpy(close)                      # (c)
            if bool((near_thr | order).any()):
                fragile.add(c)
    cut = None
    if len(ref) >= top_k or len(ours) >= top_k:
        ranked = sorted(ref, key=lambda cp: -float(probs[cp[1], cp[0]]))
        cc, cp = ranked[min(len(ranked), top_k) - 1]            # the oracle's k-th largest detection
        cut = (p64[cp, cc], pb[cp, cc])
    unexplained = []
    for c, p in diff:
        pr, b = p64[p, c], pb[p, c]
        own = abs(pr - min_score) <= b
        at_cut = cut is not None and (abs(pr - cut[0]) <= b + cut[1] or (fragile and pr <= cut[0] + b + cut[1]))
        if not (own or c in fragile or at_cut):
            unexplained.append((c, p))
    return len(diff), unexplained


def check_fused_values(out, i, loc_i, conf_i, pri):
    """Every probability and box the fused path emitted for image i lies within the per-candidate bound of the float64
    softmax and decode of the same fp32 inputs (non-finite values must be what float64 gives)."""
    k = int(out["cnt"][i])
    cls = out["cls"][i, :k].cpu().long().numpy()
    pid = out["prior"][i, :k].cpu().long().numpy()
    p64, pb = softmax_f64(conf_i.numpy())
    b64, bb = decode_f64(loc_i.numpy(), pri.numpy())
    gp = out["prob"][i, :k].cpu().double().numpy()
    gb = out["boxes"][i, :k].cpu().double().numpy()
    want_p, bound_p = p64[pid, cls], pb[pid, cls]
    bad = ~(np.abs(gp - want_p) <= bound_p)
    assert not bad.any(), (f"image {i}: {int(bad.sum())} probabilities outside their bound, e.g. {gp[bad][:3]} vs "
                           f"{want_p[bad][:3]} (bound {bound_p[bad][:3]})")
    want_b, bound_b = b64[pid], bb[pid]
    with np.errstate(invalid="ignore"):
        ok = (np.abs(gb - want_b) <= bound_b) | (gb == want_b) | (np.isnan(gb) & np.isnan(want_b))
    assert ok.all(), f"image {i}: {int((~ok).any(1).sum())} boxes outside their bound, e.g. {gb[~ok.all(1)][:2]} vs {want_b[~ok.all(1)][:2]}"


def compare_detect_with_oracle(out, loc, conf, pri, min_score, iou_thr, top_k, images):
    """The device path's detections (own softmax + decode) of ``images`` against the oracle's: every emitted probability
    and box within its bound of the float64 softmax / decode (check_fused_values), every detection that differs from
    the oracle's with a boundary proof (explain_detect_mismatches).  Returns the number of (explained) differences."""
    total = 0
    for i in images:
        rb, rc, rp, ri = O.detect_image(loc[i], conf[i], pri, min_score, iou_thr, top_k)
        k = int(out["cnt"][i])
        gi, gc = out["prior"][i, :k].cpu().long(), out["cls"][i, :k].cpu().long()
        check_fused_values(out, i, loc[i], conf[i], pri)
        ref = {(int(b), int(a)) for a, b in zip(ri, rc)}
        ours = {(int(b), int(a)) for a, b in zip(gi, gc)}
        n, unexplained = explain_detect_mismatches(loc[i], conf[i], pri, min_score, iou_thr, top_k, ours, ref)
        assert not unexplained, f"image {i}: {len(unexplained)} of {n} differing detections have no boundary proof: {unexplained[:5]}"
        total += n
    return total
