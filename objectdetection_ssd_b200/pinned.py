"""Page-locked host memory whose lifetime follows the numpy arrays that view it.

``ssdhead_host_alloc`` (cudaHostAlloc) hands back a raw pointer; numpy views built on it with ``from_address`` do not
keep anything alive by themselves.  Here every view is built on a ctypes buffer object that carries a reference to its
``PinnedBlock``, so the block is released (``ssdhead_host_free``) only when the LAST array (or slice of one) that
points into it has been collected - a caller may unpack, slice and drop the containers freely.

``StagingPool`` recycles such blocks for the per-step gt upload of ``ssd()`` (``train_function.py:62-63``,
``Losses.py:129-130``): no cudaHostAlloc / cudaFreeHost on the hot path, reuse guarded by a CUDA event recorded after
the copy that read the block.
"""
from __future__ import annotations

import ctypes as C
import threading
from typing import List, Optional, Tuple

import numpy as np

from . import _lib


class PinnedBlock:
    """One cudaHostAlloc allocation; freed when the last view dies."""

    def __init__(self, nbytes: int):
        self.lib = _lib.load()
        self.nbytes = max(int(nbytes), 16)
        self.ptr = self.lib.ssdhead_host_alloc(self.nbytes)
        if not self.ptr:
            raise RuntimeError(f"ssdhead_host_alloc({self.nbytes}) failed")

    def view(self, offset: int, count: int, dtype) -> np.ndarray:
        """1-D array of ``count`` items at byte ``offset``; the array (and everything sliced from it) owns the block."""
        dtype = np.dtype(dtype)
        nb = count * dtype.itemsize
        if offset < 0 or offset + nb > self.nbytes:
            raise ValueError("view outside the pinned block")
        buf = (C.c_uint8 * max(nb, 1)).from_address(self.ptr + offset)
        buf._owner = self                      # ndarray -> memoryview -> buf -> block
        return np.frombuffer(buf, dtype=dtype, count=count)

    def __del__(self):
        ptr, self.ptr = getattr(self, "ptr", None), None
        if ptr:
            try:
                self.lib.ssdhead_host_free(ptr)
            except Exception:                  # interpreter shutdown: the driver may already be gone
                pass


def pinned_empty(shape, dtype=np.float32) -> np.ndarray:
    """Page-locked host array (copies to and from it are asynchronous); released with its last view."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape))
    return PinnedBlock(n * dtype.itemsize).view(0, n, dtype).reshape(shape)


def gt_layout(capacity: int, B: int) -> Tuple[int, int, int, int]:
    """Byte offsets of (boxes [cap,4] f32, classes [cap] f32, offsets int32 [B+1]) in one block, 16-byte aligned, and
    the block size."""
    o1 = (capacity * 16 + 15) // 16 * 16
    o2 = o1 + (capacity * 4 + 15) // 16 * 16
    total = o2 + ((B + 1) * 4 + 15) // 16 * 16
    return 0, o1, o2, total


class Staging:
    """Packed-gt arrays inside one pinned block (so the whole batch's gt goes to the device in ONE copy)."""

    def __init__(self, capacity: int, B: int):
        self.capacity, self.B = int(capacity), int(B)
        o0, o1, o2, total = gt_layout(self.capacity, self.B)
        self.block = PinnedBlock(total)
        self.nbytes = total
        self.boxes = self.block.view(o0, self.capacity * 4, np.float32).reshape(self.capacity, 4)
        self.classes = self.block.view(o1, self.capacity, np.float32)
        self.offsets = self.block.view(o2, self.B + 1, np.int32)
        self.raw = self.block.view(0, total, np.uint8)
        self.event = None                      # torch.cuda.Event recorded after the copy that last read the block
        self.event_dev = None                  # the device of that copy's stream


class StagingPool:
    """Grow-on-demand pool of ``Staging`` blocks of one (capacity, B) class; a block is handed out again only after the
    CUDA event recorded behind its last upload has completed (normally long ago: no wait).  Host threads may share a
    pool: a block is handed to one caller at a time."""

    def __init__(self, max_free: int = 8):
        self.free: List[Staging] = []
        self.max_free = max_free
        self._lock = threading.Lock()

    def acquire(self, capacity: int, B: int, exact: bool = False) -> Staging:
        """A block for ``capacity`` gts of ``B`` images.  ``exact``: exactly that capacity, so the block has the layout
        of a device buffer made with ``gt_layout(capacity, B)`` and goes up in one copy."""
        def fits(s):
            return s.B == B and (s.capacity == capacity if exact else s.capacity >= capacity)
        oldest = None
        with self._lock:
            best: Optional[int] = None
            for i, s in enumerate(self.free):
                if fits(s) and (s.event is None or s.event.query()):
                    if best is None or s.capacity < self.free[best].capacity:
                        best = i
            if best is not None:
                return self.free.pop(best)
            for i, s in enumerate(self.free):  # everything of this shape is still in flight: wait for the oldest
                if fits(s) and len(self.free) >= self.max_free:
                    oldest = self.free.pop(i)
                    break
        if oldest is not None:
            oldest.event.synchronize()         # outside the lock: other threads keep using the pool meanwhile
            return oldest
        cap = capacity if exact else max(64, 1 << (max(capacity, 1) - 1).bit_length())   # round up: ragged batches reuse one block
        return Staging(cap, B)

    def release(self, s: Staging, event) -> None:
        s.event = event
        with self._lock:
            self.free.append(s)
            if len(self.free) > 4 * self.max_free:                     # shapes that stopped occurring
                self.free = self.free[-2 * self.max_free:]
