"""Baseline and progressive JPEG decode on the device (csrc/jpeg.cu): the file decode behind the reference's
``Image.open(path).convert('RGB')`` (utils/dataloader.py:34 through ImageFolder's loader,
utils/image_to_graph/image_to_graph_optimized.py:65-68, utils/inference.py:47), bit for bit Pillow's pixels.

    images = decode_batch(files, device)               # list of uint8 [H, W, 3] device tensors (None where unsupported)
    images = decode_batch(files, device, progressive=True)     # progressive files on the device too
    info = parse(data)                                 # host: markers -> descriptor, None = not a baseline JPEG

Only the compressed bytes cross PCIe (~14 x fewer than decoded pixels).  Files the device decoder does not cover
(progressive unless asked for, CMYK, PNG, ...) come back as ``None``; ``utils/staging.DecodePool`` decodes those with
Pillow on the host.
"""
from __future__ import annotations

import ctypes
import os
from typing import List, Optional, Sequence

import torch
from torch import Tensor

from .. import _lib, ops
from .._lib import GncJpegChain, GncJpegHuff, GncJpegImage, GncJpegScan, check

_HOST_THREADS = max(1, min(8, (os.cpu_count() or 2) - 1))


def parse(data: bytes) -> Optional[GncJpegImage]:
    """Descriptor of a baseline JPEG file, or None when the device decoder does not cover the file."""
    info = GncJpegImage()
    rc = _lib.load().gnc_jpeg_parse(data, len(data), ctypes.byref(info))
    return info if rc == _lib.GNC_OK else None


def decode_batch(datas: Sequence[bytes], device=None, staging: Optional[dict] = None,
                 progressive: bool = False) -> List[Optional[Tensor]]:
    """JPEG file contents -> ``uint8 [H, W, 3]`` tensors on ``device``, in order; ``None`` for files outside the device
    decoder's scope.  One host call parses the batch and packs descriptors and bytes into pinned memory
    (``gnc_jpeg_pack``, multi-threaded), one device call decodes it.  ``staging`` = a dict the caller keeps alive to reuse
    the pinned host buffers between calls.  ``progressive=True``: the files the baseline packer leaves out are offered
    to the progressive packer (``gnc_jpeg_pack_progressive``) and decoded by a second device call."""
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if dev.type != "cuda":
        raise RuntimeError("decode_batch decodes on a CUDA device (no CPU fallback)")
    lib = _lib.load()
    n = len(datas)
    out: List[Optional[Tensor]] = [None] * n
    if n == 0:
        return out
    staging = staging if staging is not None else {}
    if staging.get("event") is not None:
        staging["event"].synchronize()              # the previous call's copies out of the pinned buffers are done
    _decode_baseline(lib, datas, dev, staging, out)
    rest = [i for i, t in enumerate(out) if t is None] if progressive else []
    if rest:
        _decode_progressive(lib, [datas[i] for i in rest], rest, dev, staging, out)
    return out


def _decode_baseline(lib, datas, dev, staging: dict, out: list) -> list:
    n = len(datas)
    total_bytes = sum(len(d) for d in datas)
    host_stream = staging.get("stream")
    if host_stream is None or host_stream.numel() < total_bytes:
        host_stream = staging["stream"] = torch.empty(max(total_bytes, 1 << 20), dtype=torch.uint8).pin_memory()
    info_bytes = n * ctypes.sizeof(GncJpegImage)
    host_infos = staging.get("infos")
    if host_infos is None or host_infos.numel() < info_bytes:
        host_infos = staging["infos"] = torch.empty(max(info_bytes, 1 << 16), dtype=torch.uint8).pin_memory()
    ptrs = (ctypes.c_char_p * n)(*datas)
    sizes = (ctypes.c_int64 * n)(*[len(d) for d in datas])
    index = (ctypes.c_int32 * n)()
    totals = (ctypes.c_int64 * 5)()
    check(lib.gnc_jpeg_pack(ctypes.cast(ptrs, ctypes.c_void_p), ctypes.cast(sizes, ctypes.c_void_p), n, _HOST_THREADS,
                            host_stream.data_ptr(), host_stream.numel(), host_infos.data_ptr(),
                            ctypes.cast(index, ctypes.c_void_p), ctypes.cast(totals, ctypes.c_void_p)), "jpeg_pack")
    m, stream_bytes, blocks, plane, pixels = (int(v) for v in totals)
    if m == 0:
        return out
    d_stream = host_stream[:stream_bytes].to(dev, non_blocking=True)
    d_infos = host_infos[:m * ctypes.sizeof(GncJpegImage)].to(dev, non_blocking=True)
    staging["event"] = torch.cuda.Event()
    staging["event"].record()
    coef = torch.empty(64 * blocks, dtype=torch.int16, device=dev)
    planes = torch.empty(plane, dtype=torch.uint8, device=dev)
    rgb = torch.empty(3 * pixels, dtype=torch.uint8, device=dev)
    scratch = torch.empty(int(lib.gnc_jpeg_scratch_bytes(stream_bytes, m)), dtype=torch.uint8, device=dev)
    check(ops._call("jpeg_decode", 0.0, float(stream_bytes + 128 * blocks * 2 + plane * 2 + 3 * pixels),
                    lib.gnc_jpeg_decode_rgb_u8, d_stream.data_ptr(), d_infos.data_ptr(), m, blocks, pixels,
                    coef.data_ptr(), planes.data_ptr(), rgb.data_ptr(), scratch.data_ptr(), ops._stream()), "jpeg_decode")
    infos = ctypes.cast(host_infos.data_ptr(), ctypes.POINTER(GncJpegImage))
    for j in range(m):
        h, w, p0 = infos[j].height, infos[j].width, infos[j].pixel_offset
        out[index[j]] = rgb[3 * p0:3 * (p0 + h * w)].view(h, w, 3)
    return out


def _pinned(staging: dict, key: str, nbytes: int) -> Tensor:
    buf = staging.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = staging[key] = torch.empty(max(nbytes, 1 << 16), dtype=torch.uint8).pin_memory()
    return buf


def _decode_progressive(lib, datas: Sequence[bytes], where: Sequence[int], dev, staging: dict, out: list) -> None:
    """Progressive files -> ``out[where[i]]``; the files the progressive packer leaves out stay ``None``."""
    n = len(datas)
    size = ctypes.sizeof
    if staging.get("progressive_event") is not None:
        staging["progressive_event"].synchronize()
    h_stream = _pinned(staging, "progressive_stream", sum(len(d) for d in datas))
    h_frames = _pinned(staging, "progressive_frames", n * size(GncJpegImage))
    h_scans = _pinned(staging, "progressive_scans", n * _lib.GNC_JPEG_MAX_SCANS * size(GncJpegScan))
    h_chains = _pinned(staging, "progressive_chains", n * _lib.GNC_JPEG_MAX_SCANS * size(GncJpegChain))
    h_tables = _pinned(staging, "progressive_tables", n * _lib.GNC_JPEG_MAX_TABLES * size(GncJpegHuff))
    ptrs = (ctypes.c_char_p * n)(*datas)
    sizes = (ctypes.c_int64 * n)(*[len(d) for d in datas])
    index = (ctypes.c_int32 * n)()
    totals = (ctypes.c_int64 * 8)()
    check(lib.gnc_jpeg_pack_progressive(
        ctypes.cast(ptrs, ctypes.c_void_p), ctypes.cast(sizes, ctypes.c_void_p), n, _HOST_THREADS,
        h_stream.data_ptr(), h_stream.numel(), h_frames.data_ptr(), ctypes.cast(index, ctypes.c_void_p),
        h_scans.data_ptr(), h_scans.numel() // size(GncJpegScan), h_chains.data_ptr(), h_chains.numel() // size(GncJpegChain),
        h_tables.data_ptr(), h_tables.numel() // size(GncJpegHuff), ctypes.cast(totals, ctypes.c_void_p)), "jpeg_pack_progressive")
    m, stream_bytes, blocks, plane, pixels, n_scans, n_chains, n_tables = (int(v) for v in totals)
    if m == 0:
        return
    d_stream = h_stream[:stream_bytes].to(dev, non_blocking=True)
    d_frames = h_frames[:m * size(GncJpegImage)].to(dev, non_blocking=True)
    d_scans = h_scans[:n_scans * size(GncJpegScan)].to(dev, non_blocking=True)
    d_chains = h_chains[:n_chains * size(GncJpegChain)].to(dev, non_blocking=True)
    d_tables = h_tables[:n_tables * size(GncJpegHuff)].to(dev, non_blocking=True)
    staging["progressive_event"] = torch.cuda.Event()
    staging["progressive_event"].record()
    coef = torch.empty(64 * blocks, dtype=torch.int16, device=dev)
    planes = torch.empty(plane, dtype=torch.uint8, device=dev)
    rgb = torch.empty(3 * pixels, dtype=torch.uint8, device=dev)
    check(ops._call("jpeg_decode_progressive", 0.0, float(stream_bytes + 128 * blocks * 3 + plane * 2 + 3 * pixels),
                    lib.gnc_jpeg_decode_progressive_rgb_u8, d_stream.data_ptr(), d_frames.data_ptr(), m, d_scans.data_ptr(),
                    d_chains.data_ptr(), n_chains, d_tables.data_ptr(), blocks, pixels, coef.data_ptr(), planes.data_ptr(),
                    rgb.data_ptr(), ops._stream()), "jpeg_decode_progressive")
    frames = ctypes.cast(h_frames.data_ptr(), ctypes.POINTER(GncJpegImage))
    for j in range(m):
        h, w, p0 = frames[j].height, frames[j].width, frames[j].pixel_offset
        out[where[index[j]]] = rgb[3 * p0:3 * (p0 + h * w)].view(h, w, 3)
