"""Batched image -> logits pipeline: the public call for the hot path end to end.

    pipe = GraphClassifierPipeline(model, resize_value=128)
    logits = pipe.infer(images_u8)                      # [B, classes]
    loss = pipe.train_step(images_u8, labels, optimizer)
    pipe = GraphClassifierPipeline(model, 256, method="superpixel", n_segments=100, compactness=10.0)

``method``: "pixel" / "patch" grid graphs, or "superpixel" graphs of the device SLIC labels (one node per region,
graphs of different node counts in one block-diagonal batch; the model's readout pads / truncates per graph).

``images_u8`` is ``uint8 [B, r, r, 3]`` on the host (pinned or not) or on the device.
Per call: one host->device copy of the pixels (if needed), the fused graph-build
kernel, the GraphNet kernels over block-diagonal micro-batches, and - for training -
gradient accumulation across micro-batches followed by the optional cross-rank
all-reduce (utils/distributed.GradBucket) and the optimizer step.

Micro-batching bounds activation memory (SURVEY.md H3): one ``[E, 128]`` fp32 edge
tensor is 16.6 MB per resize-128 graph and the backward keeps ~4 of them per block.
"""
from __future__ import annotations

from typing import Optional

import torch
from torch import Tensor

from . import ops
from .utils.image_to_graph.batched import (build_patch_graphs, build_pixel_graphs, build_superpixel_batch,
                                           build_superpixel_batch_padded, superpixel_capacity)
from .utils.image_to_graph.slic import connectivity_min_size, slic_labels


class GraphClassifierPipeline:
    def __init__(self, model: torch.nn.Module, resize_value: int, diagonals: bool = False, method: str = "pixel",
                 patch_size: int = 8, micro_batch: Optional[int] = None, train_micro_batch: Optional[int] = None,
                 device=None, n_segments: int = 100, compactness: float = 10.0):
        self.model = model
        self.resize_value = int(resize_value)
        self.diagonals = bool(diagonals)
        self.method = method
        self.patch_size = int(patch_size)
        # superpixel graphs: the reference's slic(image, n_segments=100, compactness=10) (image_to_graph_superpixel.py:31)
        self.n_segments = int(n_segments)
        self.compactness = float(compactness)
        self.device = torch.device(device) if device is not None else next(model.parameters()).device
        if self.device.type != "cuda":
            raise RuntimeError("GraphClassifierPipeline needs the model on a CUDA device (no CPU fallback)")
        r = self.resize_value
        if method == "superpixel":
            # per-image node / edge capacities of the captured path (superpixel_capacity); E <= 6 S, three times a
            # grid node's share of edge rows, so a superpixel node is budgeted as three grid nodes
            self.superpixel_caps = superpixel_capacity(r, r, connectivity_min_size(r, r, self.n_segments))
            n = 3 * self.superpixel_caps[0]
        else:
            self.superpixel_caps = None
            n = r * r if method == "pixel" else (r // self.patch_size) ** 2
        # live fp32 activations: ~8 KB per node in inference (5 edge tensors + node tensors of
        # width 128, E ~ 2N); training peaks at ~24 KB per node (activations kept for the backward over 3 blocks plus
        # the backward's transients: 63.6 GiB measured for 171 resize-128 graphs); budget 64 GiB of the 180 GB for
        # inference and 100 GiB for training (256 resize-128 graphs per micro-batch: two per 512-graph step).
        # Superpixel graphs are small (~100 nodes): up to 1024 per call, config 4's batch in one build.
        self.micro_batch = micro_batch or max(1, min(1024 if method == "superpixel" else 512, (64 << 30) // (n * 8192)))
        self.train_micro_batch = train_micro_batch or max(1, min(256, (100 << 30) // (n * 24_000)))
        self._graphs = {}            # capture key -> (CUDAGraph, static input, static logits, static overflow flag)

    # -- staging ----------------------------------------------------------------
    def _to_device(self, images) -> Tensor:
        """``uint8 [B, r, r, 3]`` on the device.  Images of another size (one ``[B, H, W, 3]`` array, or a
        list of differently sized ``[H, W, 3]`` arrays, e.g. decoded files) are resized on the device exactly
        as the reference's ``image.resize((r, r))`` does (``ops.resize_bicubic``; a list in one
        ``ops.resize_bicubic_ragged`` call)."""
        r = self.resize_value
        if isinstance(images, (list, tuple)):
            parts = []
            for im in images:
                t = im if isinstance(im, Tensor) else torch.as_tensor(im)
                t = t if t.is_cuda else t.to(self.device, non_blocking=True)
                parts.extend([t] if t.dim() == 3 else t.unbind(0))
            return ops.resize_bicubic_ragged(parts, r, r)
        t = images if isinstance(images, Tensor) else torch.as_tensor(images)
        if t.dim() == 3:
            t = t.unsqueeze(0)
        if not t.is_cuda:
            t = t.to(self.device, non_blocking=True)
        if t.shape[1] != r or t.shape[2] != r:
            t = ops.resize_bicubic(t, r, r)
        return t

    def _build(self, images_dev: Tensor):
        if self.method == "pixel":
            return build_pixel_graphs(images_dev, diagonals=self.diagonals)
        if self.method == "patch":
            return build_patch_graphs(images_dev, patch_size=self.patch_size)
        if self.method == "superpixel":
            return build_superpixel_batch(images_dev, labels=self._labels(images_dev))
        raise ValueError(f"Unknown method: {self.method}")

    def _labels(self, images_dev: Tensor) -> Tensor:
        return slic_labels(images_dev, n_segments=self.n_segments, compactness=self.compactness)

    def _build_captured(self, images_dev: Tensor):
        """The graph build of ``infer_graphed``: ``(GraphBatch, overflow flag or None)``.  Superpixel batches take the
        padded builder there, whose sizes are known on the host; the exact one reads its output sizes back."""
        if self.method != "superpixel":
            return self._build(images_dev), None
        S_cap, E_cap = self.superpixel_caps
        return build_superpixel_batch_padded(images_dev, self._labels(images_dev), S_cap, E_cap)

    @staticmethod
    def _even_chunk(total: int, limit: int) -> int:
        """Largest chunk <= limit that splits ``total`` into equal-sized pieces (up to rounding),
        so the topology cache sees at most two distinct batch shapes."""
        n_chunks = -(-total // max(1, limit))
        return -(-total // n_chunks)

    # -- inference ----------------------------------------------------------------
    @torch.no_grad()
    def infer(self, images) -> Tensor:
        img = self._to_device(images)
        B = img.shape[0]
        outs = []
        mb = self._even_chunk(B, self.micro_batch)
        for lo in range(0, B, mb):
            gb = self._build(img[lo:lo + mb])
            out = self.model(gb.as_tuple())
            outs.append(out.reshape(1, -1) if out.dim() == 1 else out)
        return outs[0] if len(outs) == 1 else torch.cat(outs, 0)

    @torch.no_grad()
    def infer_graphed(self, images) -> Tensor:
        """Small-batch latency path - the reference classifies one image per call
        (utils/inference.py:32-71).  The whole call (graph build, GraphNet, head: ~25 launches) is
        captured once per batch shape as a CUDA graph and replayed; the pixels are copied into the
        graph's static input.  Same kernels, same results as ``infer``; the model's parameters are
        read at replay time, so updated weights are picked up, a changed architecture is not.

        Superpixel graphs (SLIC, connectivity pass, graph kernel, padded batch, CSR, GraphNet, readout and head in
        one graph) are built at the per-image capacities ``superpixel_caps``, which the pipeline's own labels cannot
        exceed; the logits are ``infer``'s, bit for bit.  This call ends in one synchronisation: it reads the
        capacity flag back.  Should it be set, the call returns ``infer(images)`` instead and counts the event in
        ``ops.SUPERPIXEL_OVERFLOW_EVENTS``."""
        t = images if isinstance(images, Tensor) else torch.as_tensor(images)
        if t.dim() == 3:
            t = t.unsqueeze(0)
        key = (tuple(t.shape), self.superpixel_caps)
        ent = self._graphs.get(key)
        if ent is None:
            if t.shape[0] > self.micro_batch:
                raise ValueError("infer_graphed is the small-batch path: use infer() for large batches")
            static_in = torch.zeros(key[0], dtype=torch.uint8, device=self.device)

            def run():
                gb, flag = self._build_captured(static_in)
                out = self.model(gb.as_tuple())
                return (out.reshape(1, -1) if out.dim() == 1 else out), flag

            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(side):        # warm-up: topology cache, kernel attributes, workspaces
                for _ in range(2):
                    run()
            torch.cuda.current_stream(self.device).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static_out, static_flag = run()
            ent = self._graphs[key] = (graph, static_in, static_out, static_flag)
        graph, static_in, static_out, static_flag = ent
        static_in.copy_(t, non_blocking=True)
        graph.replay()
        out = static_out.clone()
        if static_flag is not None and int(static_flag.item()) != 0:
            # a label map the capacities do not cover (cannot happen with the pipeline's own SLIC labels unless the
            # bound's derivation is wrong): the exact builder, same logits
            ops.SUPERPIXEL_OVERFLOW_EVENTS += 1
            return self.infer(t)
        return out

    # -- training -----------------------------------------------------------------
    def forward_backward(self, images, labels) -> Tensor:
        """Accumulates d(mean CE over this call's graphs)/d(params) into ``.grad``;
        returns the mean loss as a 0-d device tensor (no host sync)."""
        img = self._to_device(images)
        lab = labels if isinstance(labels, Tensor) else torch.as_tensor(labels)
        lab = lab.to(self.device, non_blocking=True).long()
        B = img.shape[0]
        total = torch.zeros(1, dtype=torch.float32, device=self.device)
        mb = self._even_chunk(B, self.train_micro_batch)
        # gradients that already have storage (the flat bucket, or zero_grad(set_to_none=False)) are accumulated in place
        # by the kernels that produce them (ops.ACCUMULATE_GRADS); loss, its gradient and the running total are one launch
        prev, ops.ACCUMULATE_GRADS = ops.ACCUMULATE_GRADS, True
        try:
            for lo in range(0, B, mb):
                gb = self._build(img[lo:lo + mb])
                logits = self.model(gb.as_tuple())
                loss = ops.cross_entropy(logits, lab[lo:lo + mb], scale=1.0 / B, total=total)
                loss.backward()
        finally:
            ops.ACCUMULATE_GRADS = prev
        return total.reshape(())

    def train_step(self, images, labels, optimizer, grad_bucket=None) -> Tensor:
        """One optimizer step on this rank's graphs.  ``optimizer``: ``utils.distributed.FlatAdam`` (flat parameters and
        gradients, one-launch update, doubles as the gradient bucket) or any torch optimizer, optionally with a
        ``GradBucket`` for the data-parallel all-reduce."""
        if grad_bucket is None and hasattr(optimizer, "all_reduce"):
            grad_bucket = optimizer                       # FlatAdam
        if grad_bucket is not None:
            grad_bucket.zero()
        else:
            optimizer.zero_grad(set_to_none=False)
        loss = self.forward_backward(images, labels)
        if grad_bucket is not None:
            grad_bucket.all_reduce(average=True)
        optimizer.step()
        return loss
