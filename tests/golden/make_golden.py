"""Generate tests/golden/ssd_golden.npz by running the UNMODIFIED reference (imported with the stubs of
oracle/ref_import.py) on seeded synthetic inputs.  Needs the reference sources:
SSD_REFERENCE_DIR=<reference checkout> python tests/golden/make_golden.py

What is frozen (all from the reference's own functions, nothing from the oracle or the kernels):
  priors          sha256 of the 8732x4 table + its corner form
  train  (seed 1, B=8, P=8732)   ssd() losses, class map (Losses.obj_forEach_prior___), per-image map_prior_to_bb
                                 object indices, non-zero rows of conf.grad (positives + mined), grad checksums
  ties   (hand-made gts)         class map / object map for the T1-T3 cases
  detect (seed 3, B=2, bias +8)  inference() boxes / classes / probs at min_score 0.01
  stress (seed 5, B=1, P=24564, 100 gts)  ssd() losses and class map with the prior globals overwritten
"""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from objectdetection_ssd_b200 import synth            # noqa: E402
from oracle import ref_import                          # noqa: E402
from oracle import ssd_oracle as O                     # noqa: E402  (only for the 24 564-prior table generator)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def main():
    RU, RL = ref_import.load()
    out = {}
    out["priors_sha"] = sha(RL.ancs_xywh.numpy())
    out["priors_xyxy_sha"] = sha(RL.ancs_xyxy.numpy())
    out["priors_head"] = RL.ancs_xywh[:16].numpy()

    # ---- train
    B, P = 8, 8732
    gb, gc = synth.make_gt(1, B)
    loc, conf = synth.make_head(1, B, P)
    out["train_digest"] = synth.digest(loc, conf, *gb, *gc)
    tb = [torch.from_numpy(b) for b in gb]
    tc = [torch.from_numpy(c) for c in gc]
    l = torch.from_numpy(loc).requires_grad_(True)
    c = torch.from_numpy(conf).requires_grad_(True)
    with ref_import.quiet():
        l1, l2 = RL.ssd((l, c), tc, tb)
        (l1 + l2).backward()
    cls = RL.obj_forEach_prior___.to(torch.int64)
    out["train_losses"] = np.array([l1.item(), l2.item()], np.float32)
    out["train_cls"] = cls.numpy().astype(np.uint8)
    out["train_npos"] = (cls != 20).sum(1).numpy().astype(np.int32)
    objs = []
    for i in range(B):
        j = RU.get_jaccard_tensor1(tb[i], RL.ancs_xyxy)
        _, o = RU.map_prior_to_bb(j, tc[i].clone())
        objs.append(o.numpy().astype(np.int16))
    out["train_obj_local"] = np.stack(objs)
    out["train_grad_rows"] = np.packbits((c.grad.abs().sum(-1) != 0).numpy(), axis=1)
    out["train_grad_sums"] = np.array([l.grad.abs().sum().item(), c.grad.abs().sum().item(),
                                       l.grad.sum().item(), (c.grad * torch.arange(21.)).sum().item()], np.float64)

    # ---- ties
    box = torch.tensor([[0.2, 0.2, 0.6, 0.7]])
    tb2 = [torch.cat([box, box, box]), torch.tensor([[0.5, 0.5, 0.5, 0.5], [0.1, 0.1, 0.3, 0.3]]),
           torch.tensor([[0.3, 0.3, 0.31, 0.31], [0.3, 0.3, 0.31, 0.31], [0.9, 0.9, 1.0, 1.0]])]
    tc2 = [torch.tensor([3., 7., 5.]), torch.tensor([1., 2.]), torch.tensor([0., 4., 8.])]
    tcls, tobj = [], []
    for b_, c_ in zip(tb2, tc2):
        j = RU.get_jaccard_tensor1(b_, RL.ancs_xyxy)
        cc, oo = RU.map_prior_to_bb(j, c_.clone())
        tcls.append(cc.numpy().astype(np.uint8))
        tobj.append(oo.numpy().astype(np.int16))
    out["ties_cls"] = np.stack(tcls)
    out["ties_obj"] = np.stack(tobj)

    # ---- detect
    dl, dc = synth.make_head(3, 2, P, loc_scale=0.5, bg_bias=8.0)
    out["detect_digest"] = synth.digest(dl, dc)
    for i in range(2):
        with ref_import.quiet():
            bx, cl, pr = RL.inference(torch.from_numpy(dl[i]), torch.from_numpy(dc[i]), 0, toDraw=False,
                                      min_score=0.01, iou_threshold=0.45)
        out[f"detect_boxes_{i}"] = bx.numpy()
        out[f"detect_cls_{i}"] = cl.numpy().astype(np.int32)
        out[f"detect_prob_{i}"] = pr.numpy()

    # ---- stress
    pri512 = O.make_priors(**O.SSD512)
    out["stress_priors_sha"] = sha(pri512.numpy())
    gb5, gc5 = synth.make_gt(5, 1, 100, 100)
    l5, c5 = synth.make_head(5, 1, pri512.shape[0])
    out["stress_digest"] = synth.digest(l5, c5, *gb5, *gc5)
    with ref_import.priors(RL, pri512), ref_import.quiet():
        s1, s2 = RL.ssd((torch.from_numpy(l5), torch.from_numpy(c5)), [torch.from_numpy(x) for x in gc5],
                        [torch.from_numpy(x) for x in gb5])
        scls = RL.obj_forEach_prior___.to(torch.int64)
    out["stress_losses"] = np.array([s1.item(), s2.item()], np.float32)
    out["stress_cls"] = scls.numpy().astype(np.uint8)

    out["torch_version"] = np.array(torch.__version__)
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ssd_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
