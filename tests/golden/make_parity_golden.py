"""Generate tests/golden/parity_golden.npz: what the live-reference tests compare against, frozen, so that the
comparison runs in every checkout (tests/test_parity_golden.py) and not only where the reference sources are.

    python tests/golden/make_parity_golden.py

Every value comes from the UNMODIFIED reference (oracle/ref_import.py) when its sources are available, and the file
records that as source = "reference".  Without them the values come from the oracle paths that the live tests pin to
the reference on exactly these inputs (source = "oracle"): bit for bit for the box functions, ssd() forward and
gradients (ssd_reference_style), the class map and inference(); to 1e-6 / 1e-5 for ssd_old (ssd_per_image_mean); exact
for get_map (voc_ap).  Wherever the reference is available the live tests also check the stored values against it
(tests/test_oracle_vs_reference.py, tests/test_evalmap.py), so a fixture frozen from the oracle is re-checked there.

What is frozen:
  boxes    gcxgcy_to_cxcy / xyxy_to_xywh / get_offsets_coords / get_jaccard_tensor1 on seeded inputs
  loss     (seed 11, B=4, 8732 priors) ssd() losses, class map, loc / conf gradients; ssd_old() losses
  detect   (seed 13, bias +8.5) inference() boxes / classes / probs at min_score 0.01
  map      get_map() AP per class on the seeded evaluation sets of tests/test_evalmap.py
  sgd      two SGD steps and one evaluation batch of the tiny model of tests/test_dropin_train_function.py with ssd()
           as the loss: l1 / l2 per batch and the parameter change
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from objectdetection_ssd_b200 import synth             # noqa: E402
from oracle import ref_import                           # noqa: E402
from oracle import ssd_oracle as O                      # noqa: E402
from tests.test_dropin_train_function import TinyHead, _batches, sgd_loop   # noqa: E402
from tests.test_evalmap import MAP_CASES, synth_eval    # noqa: E402

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "parity_golden.npz")


def box_inputs():
    pri = O.make_priors()
    g = torch.randn(8732, 4, generator=torch.Generator().manual_seed(3))
    bx = O.cxcywh_to_xyxy(pri)
    a = torch.rand(7, 4, generator=torch.Generator().manual_seed(4))
    a[:, 2:] = a[:, :2] + a[:, 2:] * 0.3
    return pri, g, bx, a


def loss_inputs():
    gb, gc = synth.make_gt(11, 4)
    loc, conf = synth.make_head(11, 4, 8732)
    return torch.from_numpy(loc), torch.from_numpy(conf), [torch.from_numpy(b) for b in gb], [torch.from_numpy(c) for c in gc]


def detect_inputs():
    dl, dc = synth.make_head(13, 1, 8732, loc_scale=0.5, bg_bias=8.5)
    return torch.from_numpy(dl[0]), torch.from_numpy(dc[0])


def frozen_values(live: bool) -> dict:
    """The fixture's arrays, from the reference (live) or from the oracle paths pinned to it."""
    out = {}
    pri, pxy = O.make_priors(), O.cxcywh_to_xyxy(O.make_priors())
    _, g, bx, a = box_inputs()
    loc, conf, tb, tc = loss_inputs()
    dl, dc = detect_inputs()
    l = loc.clone().requires_grad_(True)
    c = conf.clone().requires_grad_(True)
    if live:
        RU, RL = ref_import.load()
        out["box_decode"] = RU.gcxgcy_to_cxcy(g, pri).numpy()
        out["box_cxcywh"] = RU.xyxy_to_xywh(bx).numpy()
        out["box_encode"] = RU.get_offsets_coords(O.xyxy_to_cxcywh(bx)[:300], pri[100:400]).numpy()
        out["box_iou"] = RU.get_jaccard_tensor1(a, bx).numpy()
        with ref_import.quiet():
            l1, l2 = RL.ssd((l, c), tc, tb)
            (l1 + l2).backward()
            cls = RL.obj_forEach_prior___.long()
            o1, o2 = RL.ssd_old((loc, conf), tc, tb)
            db, dcl, dp = RL.inference(dl, dc, 0, toDraw=False, min_score=0.01, iou_threshold=0.45)
            maps = [[float(RU.get_map(*synth_eval(s, n))[k]) for k in range(20)] for s, n in MAP_CASES]
        ssd = lambda outputs, classes, bboxes: RL.ssd(outputs, classes, bboxes)      # noqa: E731
    else:
        out["box_decode"] = O.decode(g, pri).numpy()
        out["box_cxcywh"] = O.xyxy_to_cxcywh(bx).numpy()
        out["box_encode"] = O.encode(O.xyxy_to_cxcywh(bx)[:300], pri[100:400]).numpy()
        out["box_iou"] = O.iou_matrix(a, bx).numpy()
        l1, l2 = O.ssd_reference_style((l, c), tc, tb, pri, pxy)
        (l1 + l2).backward()
        cls = O.multibox_loss(loc, conf, tb, tc, pri, pxy)["cls"]
        o1, o2 = O.ssd_per_image_mean((loc, conf), tc, tb, pri, pxy)
        db, dcl, dp, _ = O.detect_image(dl, dc, pri, 0.01, 0.45, 200)
        maps = [list(O.voc_ap(*synth_eval(s, n))) for s, n in MAP_CASES]
        ssd = lambda outputs, classes, bboxes: O.ssd_reference_style(outputs, classes, bboxes, pri, pxy)  # noqa: E731
    out["loss_losses"] = np.array([l1.item(), l2.item()], np.float32)
    out["loss_cls"] = cls.numpy().astype(np.uint8)
    out["loss_grad_loc"] = l.grad.numpy()
    out["loss_grad_conf"] = c.grad.numpy()
    out["loss_old"] = np.array([o1.item(), o2.item()], np.float32)
    out["detect_boxes"] = db.numpy()
    out["detect_cls"] = dcl.numpy().astype(np.int32)
    out["detect_prob"] = dp.numpy()
    out["map_ap"] = np.array(maps, np.float64)
    model = TinyHead()
    start = [p.detach().clone() for p in model.parameters()]
    with ref_import.quiet():
        l12 = sgd_loop(ssd, model, torch.device("cpu"), _batches())
    out["sgd_l12"] = np.array(l12, np.float32)
    for (name, p), p0 in zip(model.named_parameters(), start):
        out[f"sgd_delta_{name}"] = (p.detach() - p0).numpy()
    return out


def main():
    live = ref_import.available()
    out = frozen_values(live)
    out["source"] = np.array("reference" if live else "oracle")
    out["torch_version"] = np.array(torch.__version__)
    np.savez_compressed(PATH, **out)
    print("wrote", PATH, os.path.getsize(PATH), "bytes, source", out["source"])


if __name__ == "__main__":
    main()
