"""The reference's OWN caller driven through the drop-in (VERDICT r1 "missing #4").

``train_function.py`` is imported UNMODIFIED (from the reference sources oracle/ref_import.py finds) with
``objectdetection_ssd_b200/dropin`` first on ``sys.path``, so its ``from Losses import *`` /
``from Util import *`` (train_function.py:3-4) bind the B200 implementation.  ``train_model`` (train_function.py:12-134)
then runs one epoch - two training iterations and one test iteration - over a tiny model that returns the
``(loc [B,8732,4], conf [B,8732,21])`` pair of Model.py:235, and the result is compared with the same loop driven by the
reference's own ``Losses.ssd`` on the CPU: printed ``l1`` / ``l2`` of both phases and every parameter after the two
SGD steps.
"""
import contextlib
import importlib
import io
import os
import re
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import ref_import
from tests import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DROPIN = os.path.join(ROOT, "objectdetection_ssd_b200", "dropin")

needs_reference = pytest.mark.skipif(not ref_import.available(), reason="unmodified reference sources not available "
                                     "(SSD_REFERENCE_DIR, or oracle/fetch_ref.py)")


@contextlib.contextmanager
def dropin_on_path():
    """dropin/ first on sys.path, then the reference directory for train_function.py itself; module table restored."""
    names = ("Losses", "Util", "train_function", "DataLists")
    saved = {k: sys.modules.pop(k, None) for k in names}
    sys.path.insert(0, ref_import.REFERENCE_DIR)
    sys.path.insert(0, DROPIN)
    try:
        yield
    finally:
        sys.path.remove(DROPIN)
        sys.path.remove(ref_import.REFERENCE_DIR)
        for k in names:
            sys.modules.pop(k, None)
            if saved[k] is not None:
                sys.modules[k] = saved[k]


class TinyHead(nn.Module):
    """Stands in for Model.py: image -> (loc [B,8732,4], conf [B,8732,21]); every parameter receives a gradient."""

    def __init__(self, P=8732):
        super().__init__()
        g = torch.Generator().manual_seed(7)
        self.conv = nn.Conv2d(3, 25, 3, padding=1)
        with torch.no_grad():
            self.conv.weight.copy_(0.2 * torch.randn(self.conv.weight.shape, generator=g))
            self.conv.bias.copy_(0.1 * torch.randn(25, generator=g))
        self.loc = nn.Parameter(0.5 * torch.randn(P, 4, generator=g))
        self.conf = nn.Parameter(torch.randn(P, 21, generator=g))

    def forward(self, x):
        f = self.conv(x).mean((2, 3))
        return (self.loc[None] * (1 + f[:, None, :4])).contiguous(), (self.conf[None] + f[:, None, 4:]).contiguous()


def _batches():
    out = {"train": [], "test": []}
    for i, (phase, B) in enumerate((("train", 4), ("train", 3), ("test", 2))):
        _, _, tb, tc = H.train_inputs(300 + i, B, 8732)
        x = torch.randn(B, 3, 8, 8, generator=torch.Generator().manual_seed(900 + i))
        out[phase].append((x, tc, tb, list(range(B))))
    return out


def sgd_loop(ssd, model, device, batches):
    """Two SGD steps (lr 0.05) with ssd() as the loss over the train batches, then the test batch without gradients;
    returns (l1, l2) of every batch."""
    model.to(device)
    opt = torch.optim.SGD(model.parameters(), lr=0.05)
    l12 = []
    for phase in ("train", "test"):
        for x, tc, tb, _ in batches[phase]:
            with torch.set_grad_enabled(phase == "train"):
                l1, l2 = ssd(model(x.to(device)), tc, tb)
            if phase == "train":
                opt.zero_grad()
                (l1 + l2).backward()
                opt.step()
            l12.append((l1.item(), l2.item()))
    return l12


def _sgd_equals_frozen(ssd, device):
    """sgd_loop with `ssd` against tests/golden/parity_golden.npz (the same loop over the reference's ssd())."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "parity_golden.npz"))
    model = TinyHead()
    start = [p.detach().clone() for p in model.parameters()]
    l12 = sgd_loop(ssd, model, device, _batches())
    assert np.allclose(l12, g["sgd_l12"], rtol=1e-5, atol=0), (l12, g["sgd_l12"])
    for (n, p), p0 in zip(model.named_parameters(), start):
        want = p0 + torch.from_numpy(g[f"sgd_delta_{n}"])
        assert torch.allclose(p.detach().cpu(), want, rtol=2e-4, atol=2e-6), n
    assert np.abs(g["sgd_delta_conf"]).max() > 1e-3, "the comparison is vacuous if the steps did not move the parameters"


def test_oracle_sgd_steps_equal_the_frozen_reference():
    from oracle import ssd_oracle as O
    pri = O.make_priors()
    pxy = O.cxcywh_to_xyxy(pri)
    _sgd_equals_frozen(lambda o, c, b: O.ssd_reference_style(o, c, b, pri, pxy), torch.device("cpu"))


@pytest.mark.gpu
def test_dropin_sgd_steps_equal_the_frozen_reference(monkeypatch):
    from objectdetection_ssd_b200 import Losses as L
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)      # the tiny conv must be fp32 on both sides
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    _sgd_equals_frozen(L.ssd, torch.device("cuda"))


@needs_reference
def test_unmodified_train_function_binds_the_dropin():
    """CPU: the import mechanics.  No compute - without a CUDA device the drop-in must refuse loudly."""
    with dropin_on_path():
        tf = importlib.import_module("train_function")
        from objectdetection_ssd_b200 import Losses as L, Util as U
        assert tf.ssd is L.ssd and tf.inference is L.inference and tf.xywh_to_xyxy is U.xywh_to_xyxy
        assert os.path.samefile(os.path.dirname(tf.__file__), ref_import.REFERENCE_DIR)
        assert tuple(tf.ancs_xywh.shape) == (8732, 4)
        if not torch.cuda.is_available():
            loc, conf, tb, tc = H.train_inputs(1, 2, 8732)
            with pytest.raises(RuntimeError, match="no CPU fallback"):
                tf.ssd((loc, conf), tc, tb)


def _run_train_model(train_model, model, device, batches, monkeypatch):
    opt = torch.optim.SGD(model.parameters(), lr=0.05)
    monkeypatch.setattr(torch, "save", lambda *a, **k: None)          # train_function.py:112 writes to a Colab path
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        model = train_model(model, opt, None, batches, {"train": 7, "test": 2}, device, 0.05, num_epochs=1)
    l12 = [(float(a), float(b)) for a, b in re.findall(r"l1 ([-\d.e+]+) , l2 ([-\d.e+]+)", buf.getvalue())]
    ep = [float(x) for x in re.findall(r"(?:train|test) Loss: ([-\d.]+)", buf.getvalue())]
    return model, l12, ep


@pytest.mark.gpu
@needs_reference
def test_train_model_through_the_dropin_equals_the_reference_loop(monkeypatch):
    RUtil, RLosses = ref_import.load()
    batches = _batches()
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)      # the tiny conv must be fp32 on both sides
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    # (a) the reference's own loop with the reference's own Losses on the CPU: its train_function module sees the
    # reference's names because ref_import put them there when it imported the pair
    saved = {k: sys.modules.get(k) for k in ("Losses", "Util", "train_function")}
    sys.modules["Losses"], sys.modules["Util"] = RLosses, RUtil
    sys.modules.pop("train_function", None)
    sys.path.insert(0, ref_import.REFERENCE_DIR)
    try:
        with ref_import.quiet():
            tf_ref = importlib.import_module("train_function")
        assert tf_ref.ssd is RLosses.ssd
        ref_model, ref_l12, ref_ep = _run_train_model(tf_ref.train_model, TinyHead(), torch.device("cpu"), batches, monkeypatch)
    finally:
        sys.path.remove(ref_import.REFERENCE_DIR)
        for k, v in saved.items():
            sys.modules.pop(k, None)
            if v is not None:
                sys.modules[k] = v
    # (b) the same unmodified train_function.py over the drop-in, on the GPU
    with dropin_on_path():
        tf = importlib.import_module("train_function")
        from objectdetection_ssd_b200 import Losses as L
        assert tf.ssd is L.ssd
        model, l12, ep = _run_train_model(tf.train_model, TinyHead(), torch.device("cuda"), batches, monkeypatch)
    assert len(l12) == 2 and len(ref_l12) == 2                           # count % 20 == 0 prints: first train + first test batch
    for (a, b), (ra, rb) in zip(l12, ref_l12):
        assert abs(a - ra) <= 1e-5 * abs(ra) and abs(b - rb) <= 1e-5 * abs(rb), (l12, ref_l12)
    for e, r in zip(ep, ref_ep):
        assert abs(e - r) <= 2e-4 * abs(r) + 1e-4                        # printed with 4 decimals
    # two SGD steps with the drop-in's gradients == two SGD steps with the reference's autograd gradients
    for (n, p), (_, q) in zip(model.named_parameters(), ref_model.named_parameters()):
        assert torch.allclose(p.detach().cpu(), q.detach(), rtol=2e-4, atol=2e-6), n
    moved = (ref_model.conf.detach() - TinyHead().conf.detach()).abs().max().item()
    assert moved > 1e-3, "the comparison is vacuous if the steps did not move the parameters"
