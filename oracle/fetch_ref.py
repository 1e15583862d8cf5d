"""Copy recipe for the UNMODIFIED reference sources (test infrastructure only).

The reference is pure Python: there is nothing to compile into ``oracle/_ref``.  What this recipe does instead is copy
the reference's seven ``*.py`` files, byte for byte, from a checkout of the reference (the argument, else
``$SSD_REFERENCE_SRC``, else ``/root/reference`` where the original project is mounted) into ``oracle/_ref/`` - a directory that is git-ignored (no reference source enters the history).
The parity tests import the unmodified ``Losses.py`` / ``Util.py`` / ``train_function.py`` from it
(``oracle/ref_import.py``), and ``bench.py --impl reference`` times the reference's own ``ssd()`` on the host cores
(``cpu_baseline.kind = "reference"``).  Nothing in the product package reads this directory.

    python oracle/fetch_ref.py <reference checkout>          # idempotent; prints what it did
"""
from __future__ import annotations

import filecmp
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DEST = os.path.join(HERE, "_ref")
FILES = ("DataLists.py", "Dataset.py", "Losses.py", "Model.py", "Util.py", "train.py", "train_function.py")


def fetch(src: str | None = None, quiet: bool = False) -> bool:
    """Returns True when ``oracle/_ref`` holds the reference afterwards."""
    src = src or os.environ.get("SSD_REFERENCE_SRC", "/root/reference")
    if not os.path.isfile(os.path.join(src, "Losses.py")):
        if not quiet:
            print(f"fetch_ref: no reference under {src}; oracle/_ref left as it is "
                  f"({'present' if os.path.isfile(os.path.join(DEST, 'Losses.py')) else 'absent'})")
        return os.path.isfile(os.path.join(DEST, "Losses.py"))
    os.makedirs(DEST, exist_ok=True)
    copied = 0
    for f in FILES:
        s, d = os.path.join(src, f), os.path.join(DEST, f)
        if os.path.isfile(s) and not (os.path.isfile(d) and filecmp.cmp(s, d, shallow=False)):
            shutil.copyfile(s, d)
            copied += 1
    if not quiet:
        print(f"fetch_ref: {copied} file(s) copied from {src} to {DEST}")
    return True


if __name__ == "__main__":
    sys.exit(0 if fetch(sys.argv[1] if len(sys.argv) > 1 else None) else 1)
