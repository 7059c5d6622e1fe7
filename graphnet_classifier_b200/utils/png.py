"""PNG decode on the device (csrc/png.cu, csrc/inflate.h): the file decode behind the reference's
``Image.open(path).convert('RGB')`` for PNG files, bit for bit Pillow's pixels.

    images = decode_batch(files, device)               # list of uint8 [H, W, 3] device tensors (None where left out)

One host call parses the batch and packs the IDAT payloads into pinned memory (``gnc_png_pack``, multi-threaded), one
device call inflates, unfilters and converts every file in two launches.  Files outside the device decoder's scope
(interlaced, APNG, iCCP / zTXt / iTXt chunks, raw data above ``GNC_PNG_MAX_RAW_BYTES``, ...) and files whose stream or
rows the device finds damaged come back as ``None``; ``utils/staging.DecodePool`` decodes those with Pillow on the host,
which gives Pillow's pixels or Pillow's exception.
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Sequence

import torch
from torch import Tensor

from .. import _lib, ops
from .._lib import GncPngImage, check
from .jpeg import _HOST_THREADS, _pinned


def decode_batch(datas: Sequence[bytes], device=None, staging: Optional[dict] = None) -> List[Optional[Tensor]]:
    """PNG file contents -> ``uint8 [H, W, 3]`` tensors on ``device``, in order; ``None`` for files the device decoder
    leaves to the host.  The per-file statuses are read back after an event synchronise on the current stream (the
    caller's copy stream in ``DecodePool.batches``), never a device-wide one.  ``staging`` = a dict the caller keeps alive
    to reuse the pinned host buffers between calls."""
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if dev.type != "cuda":
        raise RuntimeError("decode_batch decodes on a CUDA device (no CPU fallback)")
    lib = _lib.load()
    n = len(datas)
    out: List[Optional[Tensor]] = [None] * n
    if n == 0:
        return out
    staging = staging if staging is not None else {}
    size = ctypes.sizeof(GncPngImage)
    h_stream = _pinned(staging, "png_stream", sum(len(d) for d in datas))
    h_images = _pinned(staging, "png_images", n * size)
    h_status = _pinned(staging, "png_status", 4 * n)
    ptrs = (ctypes.c_char_p * n)(*datas)
    sizes = (ctypes.c_int64 * n)(*[len(d) for d in datas])
    index = (ctypes.c_int32 * n)()
    totals = (ctypes.c_int64 * 4)()
    check(lib.gnc_png_pack(ctypes.cast(ptrs, ctypes.c_void_p), ctypes.cast(sizes, ctypes.c_void_p), n, _HOST_THREADS,
                           h_stream.data_ptr(), h_stream.numel(), h_images.data_ptr(), ctypes.cast(index, ctypes.c_void_p),
                           ctypes.cast(totals, ctypes.c_void_p)), "png_pack")
    m, stream_bytes, raw_bytes, pixels = (int(v) for v in totals)
    if m == 0:
        return out
    d_stream = h_stream[:stream_bytes].to(dev, non_blocking=True)
    d_images = h_images[:m * size].to(dev, non_blocking=True)
    raw = torch.empty(raw_bytes, dtype=torch.uint8, device=dev)
    rgb = torch.empty(3 * pixels, dtype=torch.uint8, device=dev)
    status = torch.empty(m, dtype=torch.int32, device=dev)
    check(ops._call("png_decode", 0.0, float(stream_bytes + 3 * raw_bytes + 3 * pixels), lib.gnc_png_decode_rgb_u8,
                    d_stream.data_ptr(), d_images.data_ptr(), m, raw.data_ptr(), rgb.data_ptr(), status.data_ptr(),
                    ops._stream()), "png_decode")
    h_status_m = h_status[:4 * m].view(torch.int32)
    h_status_m.copy_(status, non_blocking=True)
    done = torch.cuda.Event()
    done.record()
    done.synchronize()                      # also: the pinned stream / descriptors are no longer read by the device
    images = ctypes.cast(h_images.data_ptr(), ctypes.POINTER(GncPngImage))
    st = h_status_m.tolist()
    for j in range(m):
        if st[j] == 0:
            h, w, p0 = images[j].height, images[j].width, images[j].pixel_offset
            out[index[j]] = rgb[3 * p0:3 * (p0 + h * w)].view(h, w, 3)
    return out
