"""Batched, device-resident graph construction (our extension of the reference's
one-image builders): B already-resized uint8 images in, one block-diagonal graph out
(SURVEY.md appendix A), with the CSR the model's kernels consume emitted by the same
launch - no sort, no host round trip.

The reference caches the grid edge_index per (resize, diagonals) with lru_cache
(utils/image_to_graph/image_to_graph_optimized.py:42-47); the device analogue is
``GridTopologyCache``: edge_index / CSR / positions of a (B, H, W, diagonals) batch
are built once and reused, so a steady-state step only converts pixels.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch
from torch import Tensor

from ... import _lib
from ..._lib import check
from ...ops import GraphIndex, _require_cuda, _stream, _workspace, attach_graph


@dataclass
class GraphBatch:
    """Block-diagonal batch: what ``CombinedModel.forward`` takes, plus the prebuilt
    topology.  ``edge_index`` carries ``graph`` as an attribute, so passing the plain
    triple ``(x, pos, edge_index)`` to the model keeps the fast path."""
    x: Tensor            # float32 [B*N, 3]
    pos: Tensor          # float32 [B*N, 2]
    edge_index: Tensor   # int64   [2, B*E]
    graph: GraphIndex
    num_graphs: int
    nodes_per_graph: int

    def as_tuple(self):
        return self.x, self.pos, self.edge_index


def _as_device_u8(images, device) -> Tensor:
    t = images if isinstance(images, Tensor) else torch.as_tensor(images)
    if t.dtype != torch.uint8:
        raise TypeError(f"images must be uint8, got {t.dtype}")
    if t.dim() == 3:
        t = t.unsqueeze(0)
    if t.dim() != 4 or t.shape[-1] != 3:
        raise ValueError(f"images must be [B, H, W, 3], got {tuple(t.shape)}")
    if not t.is_cuda:
        t = t.to(device, non_blocking=True)
    return t.contiguous()


def _alloc_topology(B, N, E, device, want_edge_index=True):
    i32 = dict(dtype=torch.int32, device=device)
    BE = B * E
    # zero-edge grids (1 x 1): torch reports a null data_ptr for empty tensors, so the
    # buffers are allocated with at least one element and sliced after the launch
    ei = torch.empty(2, max(BE, 1), dtype=torch.int64, device=device) if want_edge_index else None
    src = torch.empty(max(BE, 1), **i32)
    dst = torch.empty(max(BE, 1), **i32)
    drp = torch.empty(B * N + 1, **i32)
    deid = torch.empty(max(BE, 1), **i32)
    srp = torch.empty(B * N + 1, **i32)
    seid = torch.empty(max(BE, 1), **i32)
    return ei, src, dst, drp, deid, srp, seid


class GridTopologyCache:
    """(B, H, W, diagonals, patch, device) -> (pos, edge_index, GraphIndex)."""

    def __init__(self, max_entries: int = 8):
        self.max_entries = max_entries
        self._entries: dict = {}

    def get(self, key):
        return self._entries.get(key)

    def put(self, key, value):
        if len(self._entries) >= self.max_entries:
            self._entries.pop(next(iter(self._entries)))
        self._entries[key] = value


_topology_cache = GridTopologyCache()


def _build_grid(images, patch: int, diagonals: bool, device, use_cache: bool) -> GraphBatch:
    dev = torch.device(device) if device is not None else (
        images.device if isinstance(images, Tensor) and images.is_cuda else torch.device("cuda", torch.cuda.current_device()))
    img = _as_device_u8(images, dev)
    _require_cuda(img)
    B, H, W, _ = img.shape
    lib = _lib.load()
    gh, gw = (H // patch, W // patch) if patch else (H, W)
    if gh < 1 or gw < 1:
        raise ValueError("patch_size larger than the image")
    N = gh * gw
    E = int(lib.gnc_grid_num_edges(gh, gw, int(diagonals and not patch)))
    x = torch.empty(B * N, 3, dtype=torch.float32, device=dev)
    key = (B, H, W, bool(diagonals), int(patch), dev)
    cached = _topology_cache.get(key) if use_cache else None
    fn = lib.gnc_build_patch_graph_u8 if patch else lib.gnc_build_pixel_graph_u8
    fifth = int(patch) if patch else int(diagonals)
    if cached is None:
        pos = torch.empty(B * N, 2, dtype=torch.float32, device=dev)
        ei, src, dst, drp, deid, srp, seid = _alloc_topology(B, N, E, dev)
        check(fn(img.data_ptr(), B, H, W, fifth, x.data_ptr(), pos.data_ptr(), ei.data_ptr(),
                 src.data_ptr(), dst.data_ptr(), drp.data_ptr(), deid.data_ptr(), srp.data_ptr(), seid.data_ptr(),
                 _stream()), "build_graph")
        BE = B * E
        if BE == 0:
            ei, src, dst, deid, seid = ei[:, :0], src[:0], dst[:0], deid[:0], seid[:0]
        graph = GraphIndex(B * N, BE, src, dst, drp, deid, srp, seid)
        # grid edges point right / down (and along both diagonals): a node has at most one in-edge per family, which is
        # what lets the node processor's launch form the aggregated operand itself (GraphIndex.max_in_degree; an upper bound)
        graph._max_in_degree = int(gw > 1) + int(gh > 1) + (2 if (diagonals and not patch and gh > 1 and gw > 1) else 0)
        if BE > 0:
            # edge classes: every edge of a grid family has the same geometry row, so the edge
            # encoder only has to see one row per family (GraphNet._forward_tc)
            cls = torch.empty(BE, dtype=torch.int32, device=dev)
            check(lib.gnc_grid_edge_class(B, gh, gw, int(diagonals and not patch), cls.data_ptr(), _stream()),
                  "grid_edge_class")
            counts = [gh * (gw - 1), (gh - 1) * gw] + ([(gh - 1) * (gw - 1)] * 2 if (diagonals and not patch) else [0, 0])
            firsts = [0, counts[0], counts[0] + counts[1], counts[0] + counts[1] + counts[2]]
            geom = torch.zeros(4, 3, dtype=torch.float32, device=dev)
            for c in range(4):
                if counts[c] > 0:
                    rel = pos[dst[firsts[c]].long()] - pos[src[firsts[c]].long()]
                    geom[c, :2] = rel
                    geom[c, 2] = rel.abs().sum()
            graph.edge_class, graph.class_geom = cls, geom
            graph.bind_positions(pos)
            if not (diagonals and not patch):
                # at most two in-edges per node: paired destination slots for the inference path (GraphIndex.pair_slots)
                slots = torch.empty(3, 2 * B * N, dtype=torch.int32, device=dev)
                check(lib.gnc_grid_pair_slots(B, gh, gw, slots[0].data_ptr(), slots[1].data_ptr(), slots[2].data_ptr(),
                                              _stream()), "grid_pair_slots")
                graph.pair_slots = (slots[0], slots[1], slots[2])
        attach_graph(ei, graph)
        if use_cache:
            _topology_cache.put(key, (pos, ei, graph))
    else:
        pos, ei, graph = cached
        # steady state: only the pixel -> feature conversion runs
        check(fn(img.data_ptr(), B, H, W, fifth, x.data_ptr(), None, None,
                 None, None, None, None, None, None, _stream()), "build_graph")
    return GraphBatch(x, pos, ei, graph, B, N)


def build_pixel_graphs(images, diagonals: bool = False, device=None, use_cache: bool = True) -> GraphBatch:
    """uint8 ``[B, H, W, 3]`` (host or device) -> block-diagonal pixel-grid batch.
    Replaces B calls of image_to_graph_pixel_optimized + the loader's casts
    (reference image_to_graph_optimized.py:71-87, utils/dataloader.py:49-51)."""
    return _build_grid(images, 0, diagonals, device, use_cache)


def build_patch_graphs(images, patch_size: int = 8, device=None, use_cache: bool = True) -> GraphBatch:
    """Patch-graph batch (reference image_to_graph_patch.py:25-54)."""
    return _build_grid(images, int(patch_size), False, device, use_cache)


def build_superpixel_graphs(images, labels, max_nodes: Optional[int] = None, device=None):
    """Label maps -> per-image superpixel graphs (reference
    image_to_graph_superpixel.py:34-71), all images in one launch.

    Returns ``(n_nodes [B], x [B, S_max, 3], pos [B, S_max, 2], n_edges [B],
    edges [B, 2, E_max])`` on the device; entries past n_nodes / n_edges are zero.
    The SLIC segmentation that produces ``labels`` is not part of this call.
    """
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    img = _as_device_u8(images, dev)
    lab = labels if isinstance(labels, Tensor) else torch.as_tensor(labels)
    if lab.dim() == 2:
        lab = lab.unsqueeze(0)
    lab = lab.to(dev)
    B, H, W, _ = img.shape
    if tuple(lab.shape) != (B, H, W):
        raise ValueError(f"labels must be [B, H, W] = {(B, H, W)}, got {tuple(lab.shape)}")
    lo, hi = int(lab.min().item()), int(lab.max().item())
    if lo < 0:
        raise ValueError("labels must be non-negative")
    lab32 = lab.to(torch.int32).contiguous()
    S_max = int(max_nodes) if max_nodes is not None else min(hi + 1, H * W)
    E_max = S_max * (S_max - 1)
    lib = _lib.load()
    n_nodes = torch.zeros(B, dtype=torch.int32, device=dev)
    n_edges = torch.zeros(B, dtype=torch.int32, device=dev)
    x = torch.empty(B, S_max, 3, dtype=torch.float32, device=dev)
    pos = torch.empty(B, S_max, 2, dtype=torch.float32, device=dev)
    adj = torch.empty(B, S_max, S_max, dtype=torch.uint8, device=dev)
    edges = torch.empty(B, 2, max(E_max, 1), dtype=torch.int64, device=dev)
    work = _workspace(dev, B * int(lib.gnc_superpixel_workspace(S_max, hi)), torch.int32)
    check(lib.gnc_build_superpixel_graph(img.data_ptr(), lab32.data_ptr(), B, H, W, hi, S_max, max(E_max, 1),
                                         n_nodes.data_ptr(), x.data_ptr(), pos.data_ptr(), adj.data_ptr(),
                                         n_edges.data_ptr(), edges.data_ptr(), work.data_ptr(), _stream()),
          "build_superpixel_graph")
    return n_nodes, x, pos, n_edges, edges


def build_superpixel_batch(images, labels=None, n_segments: int = 100, compactness: float = 10.0,
                           max_nodes: Optional[int] = None, device=None) -> GraphBatch:
    """Superpixel graphs of a batch of images as ONE block-diagonal ``GraphBatch`` whose graphs have different node
    counts (reference image_to_graph_superpixel.py:8-73 per image): SLIC labels (``slic_labels`` unless ``labels`` is
    supplied) -> per-image graph kernel -> compaction -> CSR.  ``graph.node_ptr`` (int32 ``[B + 1]``) tells the model's
    readout where each graph's nodes are; ``nodes_per_graph`` is 0 (not constant)."""
    from .slic import slic_labels
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    img = _as_device_u8(images, dev)
    if labels is None:
        labels = slic_labels(img, n_segments=n_segments, compactness=compactness)
    n_nodes, x, pos, n_edges, edges = build_superpixel_graphs(img, labels, max_nodes=max_nodes, device=dev)
    B, S_max, E_max = x.shape[0], x.shape[1], edges.shape[2]
    lib = _lib.load()
    node_ptr = torch.empty(B + 1, dtype=torch.int32, device=dev)
    edge_ptr = torch.empty(B + 1, dtype=torch.int64, device=dev)
    check(lib.gnc_superpixel_batch_offsets(n_nodes.data_ptr(), n_edges.data_ptr(), B, S_max, E_max, node_ptr.data_ptr(),
                                           edge_ptr.data_ptr(), _stream()), "superpixel_batch_offsets")
    n_total, e_total = int(node_ptr[B].item()), int(edge_ptr[B].item())          # the one host sync: output sizes
    xb = torch.empty(n_total, 3, dtype=torch.float32, device=dev)
    pb = torch.empty(n_total, 2, dtype=torch.float32, device=dev)
    eb = torch.empty(2, e_total, dtype=torch.int64, device=dev)
    check(lib.gnc_superpixel_batch_compact(x.data_ptr(), pos.data_ptr(), edges.data_ptr(), B, S_max, E_max, node_ptr.data_ptr(),
                                           edge_ptr.data_ptr(), xb.data_ptr(), pb.data_ptr(), eb.data_ptr(), e_total, _stream()),
          "superpixel_batch_compact")
    graph = GraphIndex.from_edge_index(eb, xb.shape[0])
    graph.node_ptr = node_ptr
    attach_graph(eb, graph)
    return GraphBatch(xb, pb, eb, graph, B, 0)


def superpixel_capacity(H: int, W: int, min_size: int):
    """Per-image ``(S_cap, E_cap)``: node and directed-edge bounds of the superpixel graphs of ``slic_labels`` maps whose
    connectivity post-pass ran with ``min_size`` (``slic.connectivity_min_size``).

    Nodes: the post-pass (csrc/slic_connect.cu) keeps a 4-connected component only if it has at least ``min_size``
    pixels, except the component of pixel 0, which it always keeps; the kept components are the final labels.  Disjoint
    components of ``min_size`` pixels or more number at most ``H W // min_size``, so ``S <= H W // min_size + 1``, and
    ``S <= H W`` always (every component survives when ``min_size <= 1``).
    Edges: every final label is a 4-connected region (a dissolved component joins the component next to its first pixel),
    so contracting the regions of the pixel grid gives the region adjacency graph as a minor of a planar graph: it is
    planar and simple, with at most ``3 S - 6`` adjacent pairs (``S >= 3``), i.e. ``6 S - 12`` directed edges; with
    ``S < 3`` at most ``S (S - 1)``."""
    hw = int(H) * int(W)
    S = min(hw, hw // max(int(min_size), 1) + 1)
    return S, (S * (S - 1) if S < 3 else 6 * S - 12)


def build_superpixel_batch_padded(images, labels, S_cap: int, E_cap: int, device=None):
    """``build_superpixel_batch`` at host-known sizes, for CUDA-graph capture: no value is read back to the host.

    Returns ``(GraphBatch, overflow)``.  The batch has ``B S_cap + 1`` rows and ``B E_cap`` edges; its first
    ``node_ptr[B]`` rows and ``edge_ptr[B]`` edges are ``build_superpixel_batch``'s, in the same order; the rest are zero
    rows and self-loops on them (``gnc_superpixel_batch_padded``).  ``graph.node_ptr`` is the exact per-graph offsets,
    so the readout sees the real rows only; every real node has the same in-edges, in the same order, as in the exact
    batch, so the logits are the same bits.  ``overflow`` (int32 ``[1]`` on the device) is non-zero when an image has
    a label outside ``[0, S_cap - 1]``, more than ``S_cap`` nodes or more than ``E_cap`` edges: the batch is then not
    the exact one and its logits must not be used."""
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    img = _as_device_u8(images, dev)
    lab = labels if isinstance(labels, Tensor) else torch.as_tensor(labels)
    if lab.dim() == 2:
        lab = lab.unsqueeze(0)
    B, H, W, _ = img.shape
    if tuple(lab.shape) != (B, H, W):
        raise ValueError(f"labels must be [B, H, W] = {(B, H, W)}, got {tuple(lab.shape)}")
    S_cap, E_cap = int(S_cap), int(E_cap)
    if S_cap < 1 or E_cap < 0:
        raise ValueError("S_cap must be >= 1 and E_cap >= 0")
    lab32 = lab.to(dev, torch.int32).contiguous()
    max_label = S_cap - 1                  # labels above it are skipped by the graph kernel and flagged below
    lib = _lib.load()
    i32 = dict(dtype=torch.int32, device=dev)
    n_nodes, n_edges = torch.empty(B, **i32), torch.empty(B, **i32)
    x = torch.empty(B, S_cap, 3, dtype=torch.float32, device=dev)
    pos = torch.empty(B, S_cap, 2, dtype=torch.float32, device=dev)
    adj = torch.empty(B, S_cap, S_cap, dtype=torch.uint8, device=dev)
    edges = torch.empty(B, 2, max(E_cap, 1), dtype=torch.int64, device=dev)
    work = _workspace(dev, B * int(lib.gnc_superpixel_workspace(S_cap, max_label)), torch.int32)
    check(lib.gnc_build_superpixel_graph(img.data_ptr(), lab32.data_ptr(), B, H, W, max_label, S_cap, E_cap,
                                         n_nodes.data_ptr(), x.data_ptr(), pos.data_ptr(), adj.data_ptr(),
                                         n_edges.data_ptr(), edges.data_ptr(), work.data_ptr(), _stream()),
          "build_superpixel_graph")
    node_ptr = torch.empty(B + 1, **i32)
    edge_ptr = torch.empty(B + 1, dtype=torch.int64, device=dev)
    check(lib.gnc_superpixel_batch_offsets(n_nodes.data_ptr(), n_edges.data_ptr(), B, S_cap, E_cap, node_ptr.data_ptr(),
                                           edge_ptr.data_ptr(), _stream()), "superpixel_batch_offsets")
    N_alloc, E_alloc = B * S_cap + 1, B * E_cap
    xb = torch.empty(N_alloc, 3, dtype=torch.float32, device=dev)
    pb = torch.empty(N_alloc, 2, dtype=torch.float32, device=dev)
    eb = torch.empty(2, max(E_alloc, 1), dtype=torch.int64, device=dev)[:, :E_alloc]
    overflow = torch.empty(1, **i32)
    check(lib.gnc_superpixel_batch_padded(x.data_ptr(), pos.data_ptr(), edges.data_ptr(), n_nodes.data_ptr(),
                                          n_edges.data_ptr(), lab32.data_ptr(), B, H, W, max_label, S_cap, E_cap,
                                          node_ptr.data_ptr(), edge_ptr.data_ptr(), xb.data_ptr(), pb.data_ptr(),
                                          eb.data_ptr(), overflow.data_ptr(), _stream()), "superpixel_batch_padded")
    graph = GraphIndex.from_edge_index(eb, N_alloc, validate=False)      # every endpoint is in range by construction
    graph.node_ptr = node_ptr
    attach_graph(eb, graph)
    return GraphBatch(xb, pb, eb, graph, B, 0), overflow
