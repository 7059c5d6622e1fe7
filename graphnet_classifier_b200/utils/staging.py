"""Input staging from image FILES (SURVEY.md 8f rank 1): the reference opens one file at a time on the training thread,
``Image.open(path).convert('RGB').resize((r, r))`` (utils/dataloader.py:34 through torchvision's ImageFolder,
utils/image_to_graph/image_to_graph_optimized.py:65-70, utils/inference.py:47).  Here

* baseline JPEG files are decoded ON THE DEVICE (``utils/jpeg.py``, csrc/jpeg.cu: libjpeg's integer algorithm restated,
  bit for bit Pillow's pixels): the pool's threads only read the files and parse their markers, and only the compressed
  bytes cross PCIe; with ``device_jpeg="progressive"`` progressive JPEG files are decoded on the device too;
* with ``device_png=True`` PNG files are decoded on the device as well (``utils/png.py``, csrc/png.cu: bit for bit
  Pillow's pixels), whatever ``device_jpeg`` says about JPEG files;
* everything else (PNG unless asked for, progressive / CMYK JPEG, ...; or all files with ``device_jpeg=False``): the decode
  (``Image.open`` + ``convert('RGB')``: libjpeg inside Pillow) runs on a pool of host PROCESSES (Pillow's
  Python-level file handling holds the GIL for about half of a small file's decode time: 8 threads give 2 x one
  thread, processes scale with the cores), each image decoded straight into its slot of a shared-memory staging
  buffer that is registered with CUDA as pinned memory; PIL images that are already open (no path to hand to another
  process) are decoded on a thread pool instead;
* images of one shape travel as ONE host->device copy on a copy stream; two staging buffers alternate, so the pool
  decodes chunk ``i + 1`` while chunk ``i`` is copied and consumed;
* the resize is the Pillow-exact device kernel, so the pixels that reach the graph builder are bit for bit the
  reference's: ``ops.resize_bicubic`` when a chunk holds one shape, else one ``ops.resize_bicubic_ragged`` call over
  all its images, whatever the number of shapes.

"""
from __future__ import annotations

import os
from concurrent.futures import ThreadPoolExecutor
from typing import Iterable, Iterator, List, Optional, Sequence, Tuple

import numpy as np
import torch
from PIL import Image
from torch import Tensor

from .. import ops


_JPEG_MAGIC, _PNG_MAGIC = b"\xff\xd8", b"\x89PNG\r\n\x1a\n"


def _decode(path_or_image) -> np.ndarray:
    image = Image.open(path_or_image) if isinstance(path_or_image, (str, os.PathLike)) else path_or_image
    return np.asarray(image.convert("RGB"), dtype=np.uint8)


class _SharedPinned:
    """A shared-memory segment (visible to the worker processes by name) registered with CUDA as pinned host memory."""

    def __init__(self, nbytes: int):
        from multiprocessing import shared_memory
        self.seg = shared_memory.SharedMemory(create=True, size=int(nbytes))
        self.tensor = torch.frombuffer(self.seg.buf, dtype=torch.uint8, count=int(nbytes))
        rt = torch.cuda.cudart()
        err = rt.cudaHostRegister(self.tensor.data_ptr(), int(nbytes), 0)
        self.registered = int(err) == 0
        self.nbytes = int(nbytes)

    def close(self):
        if self.registered:
            torch.cuda.cudart().cudaHostUnregister(self.tensor.data_ptr())
            self.registered = False
        self.tensor = None
        try:
            self.seg.close()
            self.seg.unlink()
        except (BufferError, FileNotFoundError):
            pass


class DecodePool:
    """``stage(items, resize_value)`` -> ``uint8 [n, r, r, 3]`` on the device for ``items`` = file paths or PIL images.
    ``batches(items, resize_value, chunk)`` yields the same in chunks with decode / copy / compute overlapped.
    ``processes=True`` (default) decodes file paths on worker processes into shared pinned memory; PIL images and
    ``processes=False`` use the thread pool."""

    def __init__(self, workers: Optional[int] = None, device=None, processes: bool = True, slot_bytes: int = 1 << 20,
                 device_jpeg="auto", device_png: bool = False):
        self.workers = int(workers) if workers else max(1, (os.cpu_count() or 2) - 1)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.device.type != "cuda":
            raise RuntimeError("DecodePool stages onto a CUDA device (no CPU fallback)")
        self.pool = ThreadPoolExecutor(max_workers=self.workers, thread_name_prefix="gnc-decode")
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self._pinned = [None, None]             # two staging buffers (bytes), grown on demand
        self._events = [None, None]             # "buffer's last copy has finished"
        self.processes = bool(processes)
        self.slot_bytes = int(slot_bytes)       # one decoded image per slot (1 MiB holds 512 x 682 RGB; larger images come back through the pipe)
        self._procs = None
        self._shared = [None, None]
        # baseline JPEG files: Huffman + IDCT + colour on the GPU ("auto" = yes): 63 k files/s per GPU against ~1.3 k per
        # host core, only the compressed bytes cross PCIe, and the pixels are Pillow's bit for bit.  Files the device
        # decoder does not cover take the host path below either way.  "progressive": progressive files on the device too.
        self.progressive_jpeg = device_jpeg == "progressive"
        if device_jpeg == "auto":
            device_jpeg = True
        self.device_jpeg = bool(device_jpeg)
        self._jpeg_staging = [{}, {}]
        self.stats = {"device_jpeg": 0, "host_decoded": 0}
        # PNG files: inflate, unfilter and conversion on the GPU, opt-in; files the device leaves out or finds damaged
        # take the host path, which gives Pillow's pixels or Pillow's exception
        self.device_png = bool(device_png)
        self._png_staging = [{}, {}]
        if self.device_png:
            self.stats["device_png"] = 0

    def _process_pool(self):
        if self._procs is None:
            import multiprocessing as mp
            from concurrent.futures import ProcessPoolExecutor
            from . import _decode_worker
            self._procs = ProcessPoolExecutor(max_workers=self.workers, mp_context=mp.get_context("spawn"))
            list(self._procs.map(_decode_worker.warm, range(2 * self.workers)))      # start the interpreters now
        return self._procs

    def close(self) -> None:
        self.pool.shutdown(wait=True)
        if self._procs is not None:
            self._procs.shutdown(wait=True)
            self._procs = None
        torch.cuda.synchronize(self.device)
        for i, sh in enumerate(self._shared):
            if sh is not None:
                sh.close()
                self._shared[i] = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False

    # -- one chunk ---------------------------------------------------------------------
    def _staging(self, slot: int, nbytes: int) -> Tensor:
        buf = self._pinned[slot]
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8).pin_memory()
            self._pinned[slot] = buf
        return buf

    def _decode_chunk_processes(self, paths: Sequence, slot: int):
        """File paths decoded by the worker processes into slots of the shared pinned buffer; returns
        ``[(shape, indices, [pinned views [H, W, 3]])]`` grouped by shape."""
        from . import _decode_worker
        procs = self._process_pool()
        need = len(paths) * self.slot_bytes
        sh = self._shared[slot]
        if sh is None or sh.nbytes < need:
            if sh is not None:
                torch.cuda.synchronize(self.device)
                sh.close()
            try:
                sh = self._shared[slot] = _SharedPinned(max(need, 64 * self.slot_bytes))
            except OSError:                     # /dev/shm too small for the staging buffers: decode on the thread pool
                self._shared[slot] = None
                self.processes = False
                return self._decode_chunk(paths, slot)
        work = [(str(p), sh.seg.name, i * self.slot_bytes, self.slot_bytes) for i, p in enumerate(paths)]
        results = list(procs.map(_decode_worker.decode_into, work, chunksize=max(1, len(work) // (4 * self.workers))))
        groups = {}
        for i, (h, w, spill) in enumerate(results):
            n = h * w * 3
            if spill is not None:               # larger than a slot: came back through the pipe
                view = torch.from_numpy(np.ascontiguousarray(spill))
            else:
                view = sh.tensor[i * self.slot_bytes:i * self.slot_bytes + n].view(h, w, 3)
            groups.setdefault((h, w, 3), ([], []))
            groups[(h, w, 3)][0].append(i)
            groups[(h, w, 3)][1].append(view)
        return [(shape, idxs, views) for shape, (idxs, views) in groups.items()]

    def _host_decode(self, paths: Sequence) -> list:
        """Pillow on the host for the files of a device-decode chunk the device does not take: on the worker processes
        when the pool decodes JPEGs on the host (``device_jpeg=False`` with ``device_png=True``: those JPEGs stay on the
        processes they would take without ``device_png``), else on the thread pool."""
        if self.processes and not self.device_jpeg:
            from . import _decode_worker
            return list(self._process_pool().map(_decode_worker.decode, [str(p) for p in paths],
                                                 chunksize=max(1, len(paths) // (4 * self.workers))))
        return list(self.pool.map(_decode, paths))

    def _read_chunk_jpeg(self, paths: Sequence, slot: int):
        """Device-decode form of a chunk (device JPEG and / or PNG): the pool's threads read the files (the C packers
        release the GIL); files of no format the device decodes are decoded by Pillow here, on the host."""

        def read(path):
            with open(path, "rb") as f:
                return f.read()

        datas = list(self.pool.map(read, paths))
        # which files the device decoder covers is known only after the pack step (on upload); files it rejects are
        # decoded here by Pillow when their magic is not JPEG's, and after the device call otherwise
        rest = [i for i, d in enumerate(datas) if not ((self.device_jpeg and d[:2] == _JPEG_MAGIC) or
                                                        (self.device_png and d[:8] == _PNG_MAGIC))]
        host = dict(zip(rest, self._host_decode([paths[i] for i in rest]))) if rest else {}
        pairs = [(d, None) for d in datas]
        return {"jpeg": pairs, "host": host, "slot": slot, "paths": list(paths)}

    def _upload_jpeg(self, chunk, resize_value: int) -> Tensor:
        from . import jpeg as gjpeg
        r = int(resize_value)
        pairs, host = chunk["jpeg"], chunk["host"]
        datas = [d if i not in host else b"" for i, (d, _) in enumerate(pairs)]
        png = [i for i, d in enumerate(datas) if self.device_png and d[:8] == _PNG_MAGIC]
        if self.device_jpeg:
            jpeg_datas = [b"" if d[:8] == _PNG_MAGIC else d for d in datas] if png else datas
            imgs = gjpeg.decode_batch(jpeg_datas, self.device, staging=self._jpeg_staging[chunk["slot"]],
                                      progressive=self.progressive_jpeg)
        else:
            imgs = [None] * len(datas)
        n_png = 0
        if png:
            from . import png as gpng
            for i, t in zip(png, gpng.decode_batch([datas[i] for i in png], self.device,
                                                   staging=self._png_staging[chunk["slot"]])):
                imgs[i] = t
                n_png += t is not None
        late = [i for i, t in enumerate(imgs) if t is None and i not in host]     # files outside the device decoders' scope
        if late:
            host = dict(host)
            host.update(zip(late, self._host_decode([chunk["paths"][i] for i in late])))
        self.stats["device_jpeg"] += len(imgs) - len(host) - n_png
        if self.device_png:
            self.stats["device_png"] += n_png
        self.stats["host_decoded"] += len(host)
        for i, a in host.items():
            imgs[i] = torch.from_numpy(np.array(a, dtype=np.uint8)).to(self.device)
        n, shape = len(imgs), imgs[0].shape
        if all(t.shape == shape for t in imgs) and all(
                imgs[i].data_ptr() + imgs[i].numel() == imgs[i + 1].data_ptr() for i in range(n - 1)):
            batch = torch.as_strided(imgs[0], (n, *shape), (imgs[0].numel(), shape[1] * 3, 3, 1))     # already packed
            return batch if (shape[0] == r and shape[1] == r) else ops.resize_bicubic(batch, r, r)
        return ops.resize_bicubic_ragged(imgs, r, r)

    def _decode_chunk(self, items: Sequence, slot: int):
        """Decodes ``items`` on the pool; returns ``[(shape, indices, pinned view [k, H, W, 3])]`` grouped by shape."""
        if (self.device_jpeg or self.device_png) and items and all(isinstance(it, (str, os.PathLike)) for it in items):
            return self._read_chunk_jpeg(items, slot)
        if self._events[slot] is not None:
            self._events[slot].synchronize()            # the previous copy out of this buffer is done
        if self.processes and items and all(isinstance(it, (str, os.PathLike)) for it in items):
            return self._decode_chunk_processes(items, slot)
        arrays: List[np.ndarray] = list(self.pool.map(_decode, items))
        groups = {}
        for i, a in enumerate(arrays):
            groups.setdefault(a.shape, []).append(i)
        total = sum(a.nbytes for a in arrays)
        buf = self._staging(slot, total)
        out, off = [], 0
        for shape, idxs in groups.items():
            n = len(idxs) * int(np.prod(shape))
            view = buf[off:off + n].view(len(idxs), *shape)
            dst = view.numpy()

            def put(j_i, dst=dst):
                j, i = j_i
                dst[j] = arrays[i]

            list(self.pool.map(put, enumerate(idxs)))   # the copies into pinned memory are spread over the pool too
            out.append((shape, idxs, view))
            off += n
        return out

    def _upload(self, groups, slot: int, resize_value: int) -> Tensor:
        """Host->device copies on the copy stream, Pillow-exact resize on the device; returns ``[n, r, r, 3]`` in item
        order.  The caller's stream waits for the copies only."""
        if isinstance(groups, dict):
            return self._upload_jpeg(groups, resize_value)
        r = int(resize_value)
        n = sum(len(idxs) for _, idxs, _ in groups)
        cur = torch.cuda.current_stream(self.device)
        parts = []
        with torch.cuda.stream(self.copy_stream):
            for shape, idxs, view in groups:
                if isinstance(view, list):      # one pinned slot per image: gathered into a device batch by async copies
                    dev_batch = torch.empty(len(idxs), *shape, dtype=torch.uint8, device=self.device)
                    for j, v in enumerate(view):
                        dev_batch[j].copy_(v, non_blocking=True)
                    parts.append((idxs, dev_batch))
                else:
                    parts.append((idxs, view.to(self.device, non_blocking=True)))
            ev = torch.cuda.Event()
            ev.record(self.copy_stream)
        self._events[slot] = ev
        cur.wait_event(ev)
        for _, dev_imgs in parts:
            dev_imgs.record_stream(cur)
        if len(parts) == 1:
            dev_imgs = parts[0][1]
            return dev_imgs if (dev_imgs.shape[1] == r and dev_imgs.shape[2] == r) else ops.resize_bicubic(dev_imgs, r, r)
        imgs = [None] * n
        for idxs, dev_imgs in parts:
            for i, im in zip(idxs, dev_imgs):
                imgs[i] = im
        return ops.resize_bicubic_ragged(imgs, r, r)

    # -- public ------------------------------------------------------------------------
    def stage(self, items: Sequence, resize_value: int) -> Tensor:
        return self._upload(self._decode_chunk(list(items), 0), 0, resize_value)

    def _stage_async(self, items: Sequence, slot: int, resize_value: int):
        """Feeder-thread half of ``batches``: read / decode one chunk.  The device-JPEG form also packs, copies and decodes
        here, on the copy stream, so that none of a chunk's host work sits between two chunks of the consumer's GPU work."""
        torch.cuda.set_device(self.device)
        chunk = self._decode_chunk(items, slot)
        if not isinstance(chunk, dict):
            return chunk, None, None
        with torch.cuda.stream(self.copy_stream):
            px = self._upload_jpeg(chunk, resize_value)
            ev = torch.cuda.Event()
            ev.record(self.copy_stream)
        return None, px, ev

    def batches(self, items: Sequence, resize_value: int, chunk: int = 128) -> Iterator[Tensor]:
        """Chunks of ``chunk`` items as device tensors; chunk ``i + 1`` is read, decoded and (device-JPEG form) resized on
        the feeder thread / copy stream while the caller consumes chunk ``i``."""
        items = list(items)
        chunks = [items[lo:lo + chunk] for lo in range(0, len(items), chunk)]
        if not chunks:
            return
        feeder = ThreadPoolExecutor(max_workers=1, thread_name_prefix="gnc-stage")
        try:
            pending = feeder.submit(self._stage_async, chunks[0], 0, resize_value)
            for i in range(len(chunks)):
                groups, px, ev = pending.result()
                if i + 1 < len(chunks):
                    pending = feeder.submit(self._stage_async, chunks[i + 1], (i + 1) & 1, resize_value)
                if px is None:
                    yield self._upload(groups, i & 1, resize_value)
                else:
                    cur = torch.cuda.current_stream(self.device)
                    cur.wait_event(ev)
                    px.record_stream(cur)
                    yield px
        finally:
            feeder.shutdown(wait=True)


def infer_files(pipeline, paths: Iterable, pool: Optional[DecodePool] = None, chunk: Optional[int] = None) -> Tensor:
    """File paths (or PIL images) -> logits ``[n, classes]`` through ``GraphClassifierPipeline.infer``: threaded decode,
    double-buffered pinned copies, device resize, graph build and GraphNet on the stream."""
    own = pool is None
    pool = pool or DecodePool(device=pipeline.device)
    # chunk i + 1 is staged (host work + decode kernels on the copy stream) while the model runs on chunk i
    chunk = chunk or 256
    try:
        outs = [pipeline.infer(px) for px in pool.batches(list(paths), pipeline.resize_value, chunk)]
    finally:
        if own:
            pool.close()
    return outs[0] if len(outs) == 1 else torch.cat(outs, 0)
