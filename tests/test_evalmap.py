"""get_map (VOC 11-point AP, Util.py:783-885): oracle pinned against the live reference on the CPU; the GPU kernel
against the oracle (exact: integer TP/FP decisions from bit-exact IoU, fp64 precision/recall)."""
import os

import numpy as np
import pytest
import torch

from oracle import ref_import
from oracle import ssd_oracle as O


MAP_CASES = [(5, 6), (6, 25)]         # (seed, images) of the get_map comparisons with the reference


def synth_eval(seed, images, classes=4, ties=False):
    g = torch.Generator().manual_seed(seed)
    gtb, gtc, dbx, dcl, dsc = [], [], [], [], []
    for _ in range(images):
        n = int(torch.randint(1, 6, (1,), generator=g))
        c = torch.rand(n, 2, generator=g) * 0.6 + 0.2
        s = torch.rand(n, 2, generator=g) * 0.3 + 0.1
        b = torch.cat([c - s / 2, c + s / 2], 1)
        gtb.append(b)
        gtc.append(torch.randint(0, classes, (n,), generator=g).float())
        m = int(torch.randint(0, 30, (1,), generator=g))
        src = torch.randint(0, n, (m,), generator=g)
        jit = (torch.rand(m, 4, generator=g) - 0.5) * 0.15
        dbx.append(b[src] + jit)
        keep = torch.rand(m, generator=g) < 0.8
        dcl.append(torch.where(keep, gtc[-1][src], torch.randint(0, classes, (m,), generator=g).float()).long())
        sc = torch.rand(m, generator=g)
        dsc.append(torch.round(sc * 8) / 8 if ties else sc)
    return dbx, dcl, dsc, gtb, gtc


@pytest.mark.skipif(not ref_import.available(), reason="unmodified reference sources not available (SSD_REFERENCE_DIR)")
@pytest.mark.parametrize("seed,images", MAP_CASES)
def test_oracle_voc_ap_equals_reference_get_map(seed, images):
    RU, _ = ref_import.load()
    dbx, dcl, dsc, gtb, gtc = synth_eval(seed, images)
    with ref_import.quiet():
        ref = RU.get_map(dbx, dcl, dsc, gtb, gtc)
    mine = O.voc_ap(dbx, dcl, dsc, gtb, gtc)
    assert all(float(ref[c]) == mine[c] for c in range(20))
    assert mine[:4].max() > 0.1 and (mine[4:] == 0).all()      # classes without detections score 0
    # the frozen values (tests/golden/parity_golden.npz) are the reference's
    assert np.array_equal(_frozen_ap(seed, images), [float(ref[c]) for c in range(20)])


def _frozen_ap(seed, images):
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "parity_golden.npz"))
    return g["map_ap"][MAP_CASES.index((seed, images))]


@pytest.mark.gpu
@pytest.mark.parametrize("seed,images", MAP_CASES)
def test_gpu_get_map_equals_frozen_reference_get_map(seed, images):
    from objectdetection_ssd_b200 import Util
    got = Util.get_map(*synth_eval(seed, images))
    assert np.array_equal(np.array([got[c] for c in range(20)]), _frozen_ap(seed, images))


@pytest.mark.gpu
@pytest.mark.parametrize("seed,images,ties", [(5, 6, False), (7, 60, False), (8, 40, True)])
def test_gpu_get_map_equals_oracle(seed, images, ties):
    from objectdetection_ssd_b200 import Util
    dbx, dcl, dsc, gtb, gtc = synth_eval(seed, images, ties=ties)
    got = Util.get_map(dbx, dcl, dsc, gtb, gtc)
    ref = O.voc_ap(dbx, dcl, dsc, gtb, gtc)
    assert set(got) == set(range(20))
    assert np.array_equal(np.array([got[c] for c in range(20)]), ref), (got, ref)


@pytest.mark.gpu
def test_gpu_get_map_on_detect_output():
    """End of the path: detections of the batched front end scored against the gts they were generated from."""
    from objectdetection_ssd_b200 import Losses, Util
    from tests import helpers as H
    pri = H.priors()
    loc, conf, tb, tc = H.train_inputs(97, 6, pri.shape[0])
    # logits that favour the matched class on positive priors -> a detector that partly finds the gts
    ref = O.multibox_loss(loc, conf, tb, tc, pri)
    conf = conf * 0.1
    conf[..., 20] += 4.0
    for b in range(6):
        p = ref["pos"][b].nonzero().flatten()
        conf[b, p, ref["cls"][b, p]] += 9.0
        loc[b, p] = O.encode(O.xyxy_to_cxcywh(torch.cat(tb))[ref["obj"][b, p]], pri[p])
    out = Losses.inference_batch(loc.cuda(), conf.cuda(), top_k=200, min_score=0.05)
    cnt = out["cnt"].cpu()
    db = [out["boxes"][b, :int(cnt[b])].cpu() for b in range(6)]
    dc = [out["cls"][b, :int(cnt[b])].cpu().long() for b in range(6)]
    ds = [out["prob"][b, :int(cnt[b])].cpu() for b in range(6)]
    got = Util.get_map(db, dc, ds, tb, tc)
    want = O.voc_ap(db, dc, ds, tb, tc)
    assert np.array_equal(np.array([got[c] for c in range(20)]), want)
    present = sorted(set(int(x) for t in tc for x in t.tolist()))
    assert np.mean([got[c] for c in present]) > 0.5
