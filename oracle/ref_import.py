"""Import the UNMODIFIED reference for fixture generation.

TEST INFRASTRUCTURE ONLY.  The reference sources are not part of this repository:
they are read from ``$SSD_REFERENCE_DIR``, else from ``/root/reference`` where the
original project is mounted, else from the copy ``oracle/fetch_ref.py`` makes in
``oracle/_ref``.  This module is used by the fixture generators under ``tests/golden``
and by the pinning tests against the live reference (which skip where the sources
are absent; the frozen fixtures are checked everywhere).  Nothing in the product
package imports it.

The reference cannot be imported as-is in this image: ``Util.py:7,11`` import
matplotlib (not installed) and ``Util.py:14-16`` parse the VOC annotation set
from cwd-relative paths at import time.  We register empty stub modules for
``matplotlib*`` and ``DataLists`` in ``sys.modules`` (no reference source is
edited or copied), import ``Util`` / ``Losses``, then force their module-level
``device`` to CPU and patch the image-size lookup so ``inference`` returns
fractional boxes.
"""
from __future__ import annotations

import contextlib
import io
import os
import sys
import types
import warnings

_HERE = os.path.dirname(os.path.abspath(__file__))


MOUNT = "/root/reference"      # where a checkout of the original project is mounted read-only, when it is


def _default_dir() -> str:
    if os.path.isfile(os.path.join(MOUNT, "Losses.py")):
        return MOUNT
    return os.path.join(_HERE, "_ref")


REFERENCE_DIR = os.environ.get("SSD_REFERENCE_DIR") or _default_dir()


def available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_DIR, "Losses.py"))


_cached = None


def load():
    """Return ``(Util, Losses)`` modules of the reference, CPU-forced."""
    global _cached
    if _cached is not None:
        return _cached
    if not available():
        raise RuntimeError(f"reference not found under {REFERENCE_DIR}")
    import torch

    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.patches"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.modules["matplotlib"].patches = sys.modules["matplotlib.patches"]
    stub = types.ModuleType("DataLists")
    stub.call_on_load = lambda: None
    stub.all_images = {"train": ["synthetic"] * 4096, "test": ["synthetic"] * 4096}
    stub.all_multi_labels = {"train": [], "test": []}
    stub.all_multi_bboxes = {"train": [], "test": []}
    stub.all_difficulties = {"train": [], "test": []}
    saved = {k: sys.modules.get(k) for k in ("DataLists", "Util", "Losses")}
    sys.modules["DataLists"] = stub
    sys.modules.pop("Util", None)
    sys.modules.pop("Losses", None)
    sys.path.insert(0, REFERENCE_DIR)
    try:
        with warnings.catch_warnings(), contextlib.redirect_stdout(io.StringIO()):
            warnings.simplefilter("ignore")
            import Util as RUtil  # noqa: N811
            import Losses as RLosses  # noqa: N811
    finally:
        sys.path.remove(REFERENCE_DIR)
        # do not leave the reference's module names shadowing the drop-in ones
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    cpu = torch.device("cpu")
    RUtil.device = cpu
    RLosses.device = cpu
    RLosses.get_img_sz = lambda path: (1, 1)
    _cached = (RUtil, RLosses)
    return _cached


@contextlib.contextmanager
def quiet():
    """Silence the reference's progress prints (Util.py:107, Losses.py:67-85)."""
    with warnings.catch_warnings(), contextlib.redirect_stdout(io.StringIO()):
        warnings.simplefilter("ignore")
        yield


@contextlib.contextmanager
def priors(RLosses, cxcywh):
    """Temporarily replace the reference's module-global prior tables
    (read at call time: Losses.py:23,129,181) - used for the 24 564-prior case."""
    RUtil, _ = load()
    old = (RLosses.ancs_xywh, RLosses.ancs_xyxy)
    RLosses.ancs_xywh = cxcywh
    RLosses.ancs_xyxy = RUtil.xywh_to_xyxy(cxcywh)
    try:
        yield
    finally:
        RLosses.ancs_xywh, RLosses.ancs_xyxy = old
