"""Worker side of utils/staging.DecodePool's process mode.  Imports numpy and Pillow only (a spawned worker must not pay
for torch / CUDA): decodes one file, ``Image.open(path).convert('RGB')`` exactly as the reference does
(utils/dataloader.py:34 through ImageFolder's loader), straight into its slot of a shared-memory staging buffer that
the parent has registered with CUDA as pinned memory."""
from __future__ import annotations

from multiprocessing import shared_memory

import numpy as np
from PIL import Image

_open = {}          # shared-memory segments this worker has attached to, by name


def _segment(name: str):
    seg = _open.get(name)
    if seg is None:
        if len(_open) > 8:          # segments of pools that have been closed since
            for s in _open.values():
                s.close()
            _open.clear()
        seg = shared_memory.SharedMemory(name=name)
        _open[name] = seg
    return seg


def decode_into(args):
    """``(path, segment name, byte offset, slot bytes)`` -> ``(H, W, None)`` with the RGB pixels written at the offset,
    or ``(H, W, pixels)`` when the image does not fit the slot (the parent then copies them itself)."""
    path, name, offset, slot_bytes = args
    arr = np.asarray(Image.open(path).convert("RGB"), dtype=np.uint8)
    h, w = arr.shape[0], arr.shape[1]
    if arr.nbytes > slot_bytes:
        return h, w, arr
    seg = _segment(name)
    np.frombuffer(seg.buf, dtype=np.uint8, count=arr.nbytes, offset=offset)[:] = arr.reshape(-1)
    return h, w, None


def decode(path):
    """``Image.open(path).convert('RGB')`` as an array, returned through the pipe."""
    return np.asarray(Image.open(path).convert("RGB"), dtype=np.uint8)


def warm(_):
    return True
