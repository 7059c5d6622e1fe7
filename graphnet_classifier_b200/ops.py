"""Torch-facing operators over the C ABI (include/gnc.h).

torch is used for device memory, streams and autograd bookkeeping only; every
arithmetic step is a libgnc kernel.  Tensors must live on a CUDA device - there is
no CPU path (``_require_cuda`` raises).

Operators (each with its backward wired through ``torch.autograd.Function``):
  GraphIndex           int32 endpoints + stable CSR by destination and by source
  linear               act(concat(gathered segments) @ W.T + b)       models/MLP.py:24-27
  layer_norm           LayerNorm (+ residual)                          models/MLP.py:34-35, GNN.py:62,102
  aggregate            scatter_sum(edge_attr, col)                     models/GNN.py:99
  gather_rows          x[row] / x[col]                                 PyG MetaLayer, models/GNN.py:146
  edge_geometry        [pos[col]-pos[row], L1]                         models/GNN.py:299-302
  resize_bicubic       PIL Image.resize((r, r)) on the device, bit-exact  utils/image_to_graph/image_to_graph_optimized.py:65-70
  resize_bicubic_ragged  the same for a list of images of different sizes, in three launches
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence

import torch
from torch import Tensor

import os

from . import _lib
from ._lib import GncSeg, GncTcChain, GncTcEpilogue, check

# Dense engine for width-128 layers: "tc" = tcgen05 3xTF32 kernels (csrc/tc_linear.cu),
# "fp32" = CUDA-core GEMM (csrc/dense.cu).  Both meet the 1e-5 parity bar; "fp32" is the
# implementation the tensor-core path is tested against.
ENGINE = os.environ.get("GNC_ENGINE", "tc")
# Training schedule of the tensor-core engine: "core" = one autograd.Function with a hand-scheduled
# backward (tc_train.py), "opwise" = one autograd.Function per layer (what "core" is tested against).
TRAIN_PATH = os.environ.get("GNC_TRAIN_PATH", "core")
# The chained inference kernels split operands into two fp16 pieces after a FIXED power-of-two scaling: hidden activations
# of magnitude >= 4094 leave their domain and come out as inf / NaN (csrc/tc_chain.cu).  With the guard on, an inference
# forward whose node outputs are not all finite is evaluated again on the 3xTF32 per-layer engine (no such limit); the
# check costs one reduction over [N, 1] and a device->host sync, and is skipped while a CUDA graph is being captured.
# Set by GraphClassifierPipeline.forward_backward while it accumulates a step over micro-batches: the kernels that
# produce a parameter gradient then ADD it into the parameter's existing ``.grad`` (a view of the flat gradient bucket)
# and autograd receives None for it - no per-micro-batch ``grad += new`` passes (reference: ``loss.backward()`` on one
# graph per step, utils/train_model.py:41; the accumulation over micro-batches is ours).
ACCUMULATE_GRADS = False


def grad_sink(p):
    """``p.grad`` when gradients are accumulated in place and ``p`` has contiguous fp32 gradient storage, else None."""
    if not ACCUMULATE_GRADS or p is None:
        return None
    g = getattr(p, "grad", None)
    if g is None or g.dtype != torch.float32 or not g.is_contiguous() or not p.requires_grad:
        return None
    return g


CHAIN_GUARD = os.environ.get("GNC_CHAIN_GUARD", "1") != "0"
# scatter_sum folded into the node processor's launch when no node has more than two in-edges (grid graphs without
# diagonals); "0" keeps the aggregation as a launch of its own (the form the fused one is tested against)
FUSE_AGG = os.environ.get("GNC_FUSE_AGG", "1") != "0"
# Inference on grid graphs without diagonals keeps edge latents in paired destination slots (GraphIndex.pair_slots): the
# node launch reads a node's two edge rows as adjacent rows, and the last block's edge launch writes the per-node sums
# instead of edge latents (with FUSE_AGG only).  "0" keeps edge-id order (the form the slot order is tested against).
PAIRED_EDGES = os.environ.get("GNC_PAIRED_EDGES", "1") != "0"
CHAIN_GUARD_EVENTS = 0          # how many forwards took the fallback (tests, diagnostics)
# how many GraphClassifierPipeline.infer_graphed calls on superpixel graphs found a label map beyond the captured
# batch's capacities and returned the exact builder's logits instead (tests, diagnostics)
SUPERPIXEL_OVERFLOW_EVENTS = 0


def _require_cuda(*ts: Tensor) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError(
                "graphnet_classifier_b200 operators run on CUDA tensors only (sm_100a kernels, "
                "no CPU fallback); got a tensor on " + str(t.device))


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _rows(t: Tensor) -> Tensor:
    """2-D fp32 view whose rows are unit-stride (the layout every kernel expects)."""
    if t.dtype != torch.float32:
        t = t.float()
    if t.dim() != 2:
        t = t.reshape(t.shape[0], -1) if t.dim() > 0 else t.reshape(1, 1)
    if t.shape[1] > 1 and t.stride(1) != 1:
        t = t.contiguous()
    if t.shape[0] > 1 and t.stride(0) < t.shape[1]:
        t = t.contiguous()
    if t.shape[1] == 1 and t.shape[0] > 1 and t.stride(0) < 1:
        t = t.contiguous()
    return t


def _ld(t: Tensor) -> int:
    return t.stride(0) if t.shape[0] > 1 else max(t.shape[1], 1)


class KernelProfile:
    """Optional per-launch timing (CUDA events on the launching stream) used by bench.py
    to attribute step time to kernels and to compute achieved FLOP/s / GB/s live.
    Enable with ``ops.PROFILE = KernelProfile()``; ``summary()`` synchronises."""

    def __init__(self):
        self.records = []

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for name, flops, nbytes, s, e in self.records:
            d = out.setdefault(name, dict(calls=0, ms=0.0, flops=0.0, bytes=0.0))
            d["calls"] += 1
            d["ms"] += s.elapsed_time(e)
            d["flops"] += flops
            d["bytes"] += nbytes
        return out


PROFILE: Optional[KernelProfile] = None


def _call(name: str, flops: float, nbytes: float, fn, *args) -> int:
    prof = PROFILE
    if prof is None:
        return fn(*args)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    rc = fn(*args)
    e.record()
    prof.records.append((name, flops, nbytes, s, e))
    return rc


_workspaces: dict = {}


def _workspace(device, n_elems: int, dtype=torch.float32) -> Tensor:
    """Per-(device, stream, dtype) scratch buffer, grown on demand.  Kernels using it
    are ordered on the stream, so one buffer per stream is enough."""
    key = (device, _stream(), dtype)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < n_elems:
        buf = torch.empty(max(int(n_elems), 1024), dtype=dtype, device=device)
        _workspaces[key] = buf
    return buf


# ----------------------------------------------------------------------------
# graph index
# ----------------------------------------------------------------------------
class GraphIndex:
    """Topology of a (batched) graph as the kernels consume it: int32 endpoints and
    the stable CSR of edge ids by destination (in-edges, ascending edge id - the CPU
    reference's summation order) and by source."""

    __slots__ = ("num_nodes", "num_edges", "src", "dst", "dst_rowptr", "dst_eid", "src_rowptr", "src_eid",
                 "edge_class", "class_geom", "pos_ref", "pos_version", "class_sum_plan", "node_ptr", "_max_in_degree",
                 "pair_slots")

    def __init__(self, num_nodes, num_edges, src, dst, dst_rowptr, dst_eid, src_rowptr, src_eid):
        self.num_nodes, self.num_edges = int(num_nodes), int(num_edges)
        self.src, self.dst = src, dst
        self.dst_rowptr, self.dst_eid = dst_rowptr, dst_eid
        self.src_rowptr, self.src_eid = src_rowptr, src_eid
        # Optional (grid builders): edges fall into a few classes with identical geometry rows
        # [pos[dst]-pos[src], L1] (SURVEY.md 0.4).  ``edge_class`` int32 [E], ``class_geom`` float
        # [n_classes, P+1]; valid only together with the very ``pos`` tensor the builder emitted
        # (``pos_ref``), which is what the model checks before taking the table shortcut.
        self.edge_class = None
        self.class_geom = None
        self.pos_ref = None
        self.pos_version = -1           # pos_ref._version when the classes were derived from it
        self.class_sum_plan = None      # lazily built CSRs for per-class gradient sums (tc_train.class_sum_plan)
        # int32 [B + 1] node offsets of a batch whose graphs have DIFFERENT node counts (superpixel graphs); None for
        # fixed-size batches, where graph b owns rows b * num_nodes .. (b + 1) * num_nodes - 1
        self.node_ptr = None
        self._max_in_degree = None      # largest in-degree (lazy; builders that know it set it)
        # Optional (grid builders, no diagonals): (src, dst, class) int32 [2 * num_nodes] of the paired destination slots -
        # slot 2v holds node v's in-edge with the smaller edge id, slot 2v + 1 the other; src = -1 marks a slot without an
        # edge (gnc_grid_pair_slots).  Edge latents in this row order need no index to be summed per node.
        self.pair_slots = None

    def max_in_degree(self) -> int:
        """Largest number of edges arriving at one node: with at most two, the node processor's launch forms the
        aggregated operand itself (``tc_mlp_chain(agg=...)``).  One device reduction per topology, cached."""
        if self._max_in_degree is None:
            if torch.cuda.is_current_stream_capturing():
                return 1 << 30          # unknown and no synchronisation allowed here: callers take the general path
            rp = self.dst_rowptr
            self._max_in_degree = int((rp[1:] - rp[:-1]).max().item()) if rp.numel() > 1 else 0
        return self._max_in_degree

    def bind_positions(self, pos: Tensor) -> None:
        """Remember the ``pos`` tensor (and its in-place version) the edge classes were derived from."""
        self.pos_ref, self.pos_version = pos, pos._version

    def classes_valid_for(self, pos: Tensor) -> bool:
        """True when ``pos`` is the very tensor the builder emitted with this topology AND it has not been edited in
        place since (jitter / normalisation bump ``_version``): only then does the per-class geometry table describe
        the edges, otherwise the model takes the generic per-edge path."""
        return (self.edge_class is not None and self.pos_ref is pos and pos._version == self.pos_version)

    @staticmethod
    def from_edge_index(edge_index: Tensor, num_nodes: int, validate: bool = True) -> "GraphIndex":
        """Stable counting-sort CSR of an arbitrary int64 ``[2, E]`` edge_index (any
        strides - the reference hands over a transposed view, SURVEY.md 8a row a1)."""
        _require_cuda(edge_index)
        if edge_index.dtype != torch.int64:
            edge_index = edge_index.long()
        if edge_index.dim() != 2 or edge_index.shape[0] != 2:
            raise ValueError(f"edge_index must be [2, E], got {tuple(edge_index.shape)}")
        E = int(edge_index.shape[1])
        N = int(num_nodes)
        dev = edge_index.device
        lib = _lib.load()
        i32 = dict(dtype=torch.int32, device=dev)
        out = []
        bad = torch.zeros(1, **i32)
        work = _workspace(dev, int(lib.gnc_csr_workspace(N)), torch.int32)
        for k in (0, 1):
            rowptr = torch.empty(N + 1, **i32)
            eid = torch.empty(max(E, 1), **i32)[:E]
            key32 = torch.empty(max(E, 1), **i32)[:E]
            row = edge_index[k]
            stride = row.stride(0) if E > 1 else 1
            check(lib.gnc_csr_build(row.data_ptr(), stride, E, N, rowptr.data_ptr(), eid.data_ptr(),
                                    key32.data_ptr(), work.data_ptr(), bad.data_ptr(), _stream()), "csr_build")
            out.append((key32, rowptr, eid))
        if validate and int(bad.item()) != 0:
            raise IndexError(f"edge_index has node ids outside [0, {N})")
        (src, srp, seid), (dst, drp, deid) = out
        return GraphIndex(N, E, src, dst, drp, deid, srp, seid)


def attach_graph(edge_index: Tensor, graph: GraphIndex) -> Tensor:
    """Remember the prebuilt CSR on the edge_index tensor object so that a model
    called with the reference signature ``forward(x, pos, edge_index)`` finds it."""
    edge_index._gnc_graph = graph
    return edge_index


def graph_of(edge_index: Tensor, num_nodes: int) -> GraphIndex:
    g = getattr(edge_index, "_gnc_graph", None)
    if g is not None and g.num_nodes == num_nodes and g.num_edges == edge_index.shape[1]:
        return g
    return GraphIndex.from_edge_index(edge_index, num_nodes)


# ----------------------------------------------------------------------------
# raw kernel wrappers (no autograd)
# ----------------------------------------------------------------------------
def _agg_raw(rowptr: Tensor, eid: Tensor, src: Tensor, n_rows: int, out: Optional[Tensor] = None,
             accumulate: bool = False) -> Tensor:
    src = _rows(src)
    D = src.shape[1]
    if out is None:
        out = torch.empty(n_rows, D, dtype=torch.float32, device=src.device)
        accumulate = False
    E = int(eid.shape[0])
    nbytes = 4.0 * (E * D + E + (n_rows + 1) + n_rows * D)          # SURVEY.md 8d: messages + eid + rowptr + out
    check(_call("agg_csr_sum", 0.0, nbytes, _lib.load().gnc_agg_csr_sum_f32, rowptr.data_ptr(), _p(eid),
                src.data_ptr(), _ld(src), n_rows, D, out.data_ptr(), _ld(out), int(accumulate), _stream()),
          "agg_csr_sum")
    return out


def _agg_pair_raw(rowptr_a: Tensor, eid_a: Tensor, rowptr_b: Tensor, eid_b: Tensor, src: Tensor, n_rows: int):
    """``(_agg_raw(rowptr_a, eid_a, src), _agg_raw(rowptr_b, eid_b, src))`` in one launch: ``src`` comes from DRAM once."""
    src = _rows(src)
    D = src.shape[1]
    out = torch.empty(2, n_rows, D, dtype=torch.float32, device=src.device)
    E = int(eid_a.shape[0])
    nbytes = 4.0 * (E * D + 2 * E + 2 * (n_rows + 1) + 2 * n_rows * D)
    check(_call("agg_csr_sum_pair", 0.0, nbytes, _lib.load().gnc_agg_csr_sum_pair_f32, rowptr_a.data_ptr(), _p(eid_a),
                out[0].data_ptr(), rowptr_b.data_ptr(), _p(eid_b), out[1].data_ptr(), src.data_ptr(), _ld(src), n_rows, D,
                _ld(out[0]), _stream()), "agg_csr_sum_pair")
    return out[0], out[1]


def _gather_raw(src: Tensor, idx: Tensor, out: Optional[Tensor] = None, accumulate: bool = False) -> Tensor:
    src = _rows(src)
    M, D = int(idx.shape[0]), src.shape[1]
    if out is None:
        out = torch.empty(M, D, dtype=torch.float32, device=src.device)
        accumulate = False
    nbytes = 4.0 * (src.shape[0] * D + M + M * D)
    check(_call("gather_rows", 0.0, nbytes, _lib.load().gnc_gather_rows_f32, src.data_ptr(), _ld(src),
                idx.data_ptr(), M, D, out.data_ptr(), _ld(out), int(accumulate), _stream()), "gather_rows")
    return out


def _check_linear_operands(srcs: Sequence[Tensor], W: Tensor, b: Optional[Tensor], what: str) -> None:
    """The reference's ``nn.Linear`` raises on a width mismatch (models/MLP.py:24-27 via F.linear); the kernels derive K
    from the segments and read raw fp32 pointers, so the same conditions are checked here instead of computing on a
    prefix of ``W`` or on reinterpreted bytes."""
    if W.dim() != 2:
        raise RuntimeError(f"{what}: weight must be 2-D, got {tuple(W.shape)}")
    if W.dtype != torch.float32 or (b is not None and b.dtype != torch.float32):
        raise RuntimeError(f"{what}: float32 parameters only (got weight {W.dtype}"
                           f"{', bias ' + str(b.dtype) if b is not None else ''}); MLP.forward computes in float "
                           "(reference models/MLP.py:46)")
    k = sum(int(s.shape[1]) if s.dim() == 2 else int(s.numel() // max(s.shape[0], 1)) for s in srcs)
    if k != W.shape[1]:
        raise RuntimeError(f"{what}: mat1 and mat2 shapes cannot be multiplied (input width {k}, weight {tuple(W.shape)})")
    if b is not None and b.numel() != W.shape[0]:
        raise RuntimeError(f"{what}: bias has {b.numel()} elements, weight has {W.shape[0]} rows")
    for t in list(srcs) + ([b] if b is not None else []):
        if t.device != W.device:
            raise RuntimeError(f"{what}: operands on different devices ({t.device} vs {W.device})")


def _make_segs(srcs: Sequence[Tensor], idxs: Sequence[Optional[Tensor]]):
    arr = (GncSeg * len(srcs))()
    for i, (s, ix) in enumerate(zip(srcs, idxs)):
        arr[i].base = s.data_ptr()
        arr[i].idx = None if ix is None else ix.data_ptr()
        arr[i].ld = _ld(s)
        arr[i].width = s.shape[1]
    return arr


def _is_narrowk(srcs, idxs, W) -> bool:
    """Thin first layer (K <= 8, one plain segment, N % 4 == 0): streaming kernels in csrc/narrow.cu."""
    return len(srcs) == 1 and idxs[0] is None and W.shape[1] <= 8 and W.shape[0] % 4 == 0


def _linear_fwd_raw(srcs, idxs, M, W, b, relu) -> Tensor:
    N = W.shape[0]
    Y = torch.empty(M, N, dtype=torch.float32, device=W.device)
    if _is_narrowk(srcs, idxs, W):
        X, K = srcs[0], W.shape[1]
        check(_call("linear_narrowk_fwd", 2.0 * M * N * K, 4.0 * (M * K + M * N), _lib.load().gnc_linear_narrowk_fwd_f32,
                    X.data_ptr(), _ld(X), M, K, W.data_ptr(), W.stride(0), _p(b), N, int(relu), Y.data_ptr(), _ld(Y),
                    _stream()), "linear_narrowk_fwd")
        return Y
    segs = _make_segs(srcs, idxs)
    K = W.shape[1]
    lib = _lib.load()
    n_work = lib.gnc_linear_fwd_splitk_workspace(M, N, K) if K >= 2048 else 0
    if n_work > 0:      # few output tiles, long reduction (the classifier head's fc1): split K over CTAs
        work = _workspace(W.device, n_work)
        check(_call("linear_fwd", 2.0 * M * N * K, 4.0 * (M * K + N * K + M * N), lib.gnc_linear_fwd_splitk_f32,
                    segs, len(srcs), M, W.data_ptr(), W.stride(0), _p(b), N, int(relu), Y.data_ptr(), _ld(Y),
                    work.data_ptr(), work.numel(), _stream()), "linear_fwd_splitk")
        return Y
    check(_call("linear_fwd", 2.0 * M * N * K, 4.0 * (M * K + N * K + M * N), _lib.load().gnc_linear_fwd_f32,
                segs, len(srcs), M, W.data_ptr(), W.stride(0), _p(b), N, int(relu), Y.data_ptr(), _ld(Y), _stream()),
          "linear_fwd")
    return Y


class _LinearFn(torch.autograd.Function):
    """y = act(concat_s(src_s[idx_s]) @ W.T + b).  ``meta`` = per segment
    (idx int32 | None, (rowptr, eid) of the CSR grouping rows by idx | None, n_src_rows)."""

    @staticmethod
    def forward(ctx, W, b, relu, meta, *srcs):
        srcs = tuple(_rows(s) for s in srcs)
        idxs = [m[0] for m in meta]
        M = int(idxs[0].shape[0]) if idxs[0] is not None else srcs[0].shape[0]
        Wc = W if W.stride(1) == 1 else W.contiguous()
        Y = _linear_fwd_raw(srcs, idxs, M, Wc, b, relu)
        ctx.relu, ctx.meta, ctx.M = bool(relu), meta, M
        ctx.has_bias = b is not None
        ctx.W_param, ctx.b_param = W, b            # for in-place gradient accumulation (grad_sink)
        ctx.save_for_backward(Wc, Y if relu else None, *srcs)
        return Y

    @staticmethod
    def backward(ctx, dY):
        Wc, Y, *srcs = ctx.saved_tensors
        lib = _lib.load()
        dev = dY.device
        M, N, K = ctx.M, Wc.shape[0], Wc.shape[1]
        dY = _rows(dY)
        need_W, need_b = ctx.needs_input_grad[0], ctx.needs_input_grad[1] and ctx.has_bias
        # in-place accumulation into existing .grad storage (both or neither, so one flag serves the kernels)
        gW, gb = grad_sink(ctx.W_param) if need_W else None, grad_sink(ctx.b_param) if need_b else None
        acc = (gW is not None or not need_W) and (gb is not None or not need_b) and (need_W or need_b) \
            and (gW is None or (gW.dim() == 2 and gW.shape == Wc.shape))
        if not acc:
            gW = gb = None
        if (_is_narrowk(srcs, [m[0] for m in ctx.meta], Wc) and N <= 128 and not ctx.needs_input_grad[4]
                and dY.stride(0) % 4 == 0):
            # thin first layer: ReLU mask + bias gradient + weight gradient in one pass, no data gradient
            dW = (gW if acc else torch.empty(N, K, dtype=torch.float32, device=dev)) if need_W else None
            db = (gb if acc else torch.empty(N, dtype=torch.float32, device=dev)) if need_b else None
            ws_n = int(lib.gnc_linear_narrowk_wgrad_workspace(M, N, K))
            ws = _workspace(dev, ws_n)
            X = srcs[0]
            check(_call("linear_narrowk_wgrad", 2.0 * M * N * K, 4.0 * M * (N * (2 if ctx.relu else 1) + K),
                        lib.gnc_linear_narrowk_wgrad_f32, dY.data_ptr(), _ld(dY), _p(Y) if ctx.relu else None,
                        _ld(Y) if ctx.relu else 0, X.data_ptr(), _ld(X), M, N, K, _p(dW), K, _p(db), int(acc),
                        ws.data_ptr(), ws_n, _stream()), "linear_narrowk_wgrad")
            return (None, None, None, None, None) if acc else (dW, db, None, None, None)
        # bias + ReLU backward: dZ = dY * (Y > 0), db = column sums
        dZ, db = dY, None
        if ctx.relu or need_b:
            if ctx.relu:
                dZ = torch.empty(M, N, dtype=torch.float32, device=dev)
            db = (gb if acc else torch.empty(N, dtype=torch.float32, device=dev)) if need_b else None
            ws_n = int(lib.gnc_colsum_workspace(M, N))
            ws = _workspace(dev, ws_n)
            check(_call("relu_bwd_colsum", 0.0, 4.0 * M * N * (3 if ctx.relu else 1), lib.gnc_relu_bwd_colsum_f32,
                        dY.data_ptr(), _ld(dY), _p(Y) if ctx.relu else None, _ld(Y) if ctx.relu else 0, M, N,
                        dZ.data_ptr() if ctx.relu else None, _ld(dZ), _p(db), int(acc), ws.data_ptr(), ws_n, _stream()),
                  "relu_bwd_colsum")
        dW = None
        if need_W:
            dW = gW if acc else torch.empty(N, K, dtype=torch.float32, device=dev)
            segs = _make_segs(srcs, [m[0] for m in ctx.meta])
            ws_n = int(lib.gnc_linear_wgrad_workspace(M, N, K))
            ws = _workspace(dev, ws_n)
            check(_call("linear_wgrad", 2.0 * M * N * K, 4.0 * (M * K + M * N + N * K), lib.gnc_linear_wgrad_f32,
                        dZ.data_ptr(), _ld(dZ), M, N, segs, len(srcs), dW.data_ptr(), K, int(acc), ws.data_ptr(), ws_n,
                        _stream()), "linear_wgrad")
        dsrcs = []
        k0 = 0
        for i, s in enumerate(srcs):
            w = s.shape[1]
            g = None
            if ctx.needs_input_grad[4 + i]:
                dX = torch.empty(M, w, dtype=torch.float32, device=dev)
                Wv = Wc[:, k0:k0 + w]
                check(_call("linear_dgrad", 2.0 * M * N * w, 4.0 * (M * N + N * w + M * w), lib.gnc_linear_dgrad_f32,
                            dZ.data_ptr(), _ld(dZ), M, N, Wv.data_ptr(), Wc.stride(0), w, dX.data_ptr(), w, 0,
                            _stream()), "linear_dgrad")
                idx, csr, n_src = ctx.meta[i]
                if idx is None:
                    g = dX
                else:
                    # backward of the row gather = ordered segmented sum over the CSR of idx
                    g = _agg_raw(csr[0], csr[1], dX, n_src)
            dsrcs.append(g)
            k0 += w
        if acc:
            dW = db = None
        return (dW, db, None, None, *dsrcs)


def linear(srcs: Sequence[Tensor], W: Tensor, b: Optional[Tensor], relu: bool = False,
           gathers: Optional[Sequence] = None) -> Tensor:
    """``gathers[i]`` is None (rows used as is) or (idx32, (rowptr, eid), n_src_rows)."""
    _require_cuda(W, *srcs)
    _check_linear_operands(srcs, W, b, "linear")
    if gathers is None:
        gathers = [None] * len(srcs)
    meta = tuple((None, None, 0) if g is None else g for g in gathers)
    return _LinearFn.apply(W, b, relu, meta, *srcs)


class _LayerNormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, z, gamma, beta, eps, res):
        z = _rows(z)
        M, D = z.shape
        dev = z.device
        y = torch.empty(M, D, dtype=torch.float32, device=dev)
        mean = torch.empty(M, dtype=torch.float32, device=dev)
        rstd = torch.empty(M, dtype=torch.float32, device=dev)
        r = _rows(res) if res is not None else None
        check(_call("layernorm_fwd", 0.0, 4.0 * M * D * (3 if r is not None else 2), _lib.load().gnc_layernorm_fwd_f32,
                    z.data_ptr(), _ld(z), M, D, gamma.data_ptr(), beta.data_ptr(), float(eps), _p(r),
                    _ld(r) if r is not None else 0, y.data_ptr(), _ld(y), mean.data_ptr(), rstd.data_ptr(), _stream()),
              "layernorm_fwd")
        ctx.save_for_backward(z, mean, rstd, gamma)
        ctx.has_res = res is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        z, mean, rstd, gamma = ctx.saved_tensors
        lib = _lib.load()
        M, D = z.shape
        dev = z.device
        dy = _rows(dy)
        dz = torch.empty(M, D, dtype=torch.float32, device=dev)
        need_g, need_b = ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        dg = torch.empty(D, dtype=torch.float32, device=dev) if need_g else None
        db = torch.empty(D, dtype=torch.float32, device=dev) if need_b else None
        ws_n = int(lib.gnc_layernorm_bwd_workspace(M, D))
        ws = _workspace(dev, ws_n)
        check(_call("layernorm_bwd", 0.0, 4.0 * M * D * 3, lib.gnc_layernorm_bwd_f32, dy.data_ptr(), _ld(dy),
                    z.data_ptr(), _ld(z), mean.data_ptr(), rstd.data_ptr(), gamma.data_ptr(), M, D, dz.data_ptr(),
                    _ld(dz), _p(dg), _p(db), 0, ws.data_ptr(), ws_n, _stream()), "layernorm_bwd")
        return dz, dg, db, None, (dy if ctx.has_res else None)


def layer_norm(z: Tensor, gamma: Tensor, beta: Tensor, eps: float = 1e-5, res: Optional[Tensor] = None) -> Tensor:
    _require_cuda(z, gamma, beta, res)
    return _LayerNormFn.apply(z, gamma, beta, eps, res)


class _AggregateFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, e, rowptr, eid, idx, n_rows):
        ctx.save_for_backward(idx)
        return _agg_raw(rowptr, eid, e, n_rows)

    @staticmethod
    def backward(ctx, dout):
        (idx,) = ctx.saved_tensors
        return _gather_raw(dout, idx), None, None, None, None


def aggregate(edge_attr: Tensor, graph: GraphIndex) -> Tensor:
    """scatter_sum(edge_attr, col, dim=0, dim_size=N): ordered CSR segmented sum."""
    _require_cuda(edge_attr)
    return _AggregateFn.apply(edge_attr, graph.dst_rowptr, graph.dst_eid, graph.dst, graph.num_nodes)


class _GatherFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, idx, rowptr, eid):
        ctx.save_for_backward(rowptr, eid)
        ctx.n = x.shape[0]
        return _gather_raw(x, idx)

    @staticmethod
    def backward(ctx, dout):
        rowptr, eid = ctx.saved_tensors
        return _agg_raw(rowptr, eid, dout, ctx.n), None, None, None


def gather_rows(x: Tensor, idx: Tensor, rowptr: Tensor, eid: Tensor) -> Tensor:
    """x[idx]; (rowptr, eid) is the CSR grouping positions by idx (for the backward)."""
    _require_cuda(x, idx)
    return _GatherFn.apply(x, idx, rowptr, eid)


def gather_add_rows(tables: Sequence[Tensor], idxs: Sequence[Optional[Tensor]], bias: Optional[Tensor] = None,
                    relu: bool = False) -> Tensor:
    """``act(sum_s tables[s][idxs[s]] + bias)`` - up to four tables (row-gathered, or taken row by row when their
    index is None) summed in one streaming pass (no autograd)."""
    _require_cuda(*tables)
    tabs = [_rows(t) for t in tables]
    M = int(next(i.shape[0] for i in idxs if i is not None)) if any(i is not None for i in idxs) else tabs[0].shape[0]
    D = tabs[0].shape[1]
    out = torch.empty(M, D, dtype=torch.float32, device=tabs[0].device)
    n = len(tabs)
    tp = (ctypes.c_void_p * n)(*[t.data_ptr() for t in tabs])
    ip = (ctypes.c_void_p * n)(*[None if i is None else i.data_ptr() for i in idxs])
    ld = (ctypes.c_int64 * n)(*[_ld(t) for t in tabs])
    nbytes = 4.0 * (M * D + sum(t.shape[0] * D for t in tabs) + M * sum(i is not None for i in idxs))
    check(_call("gather_add_rows", 0.0, nbytes, _lib.load().gnc_gather_add_rows_f32, tp, ip, ld, n, _p(bias), int(relu),
                M, D, out.data_ptr(), _ld(out), _stream()), "gather_add_rows")
    return out


def edge_geometry(pos: Tensor, graph: GraphIndex) -> Tensor:
    _require_cuda(pos)
    if pos.requires_grad:
        raise NotImplementedError("gradients with respect to node positions are not part of this path")
    pos = _rows(pos).contiguous()
    P = pos.shape[1]
    out = torch.empty(graph.num_edges, P + 1, dtype=torch.float32, device=pos.device)
    check(_call("edge_geometry", 0.0, 4.0 * graph.num_edges * (2 + 2 * P + P + 1), _lib.load().gnc_edge_geometry_f32,
                pos.data_ptr(), P, graph.src.data_ptr(), graph.dst.data_ptr(), graph.num_edges, out.data_ptr(),
                _stream()), "edge_geometry")
    return out


_resize_tables: dict = {}


def _resize_axis_tables(in_size: int, out_size: int, device):
    """Device copies of Pillow's coefficient tables for one axis, cached per (in, out, device) - the same
    role as the reference's ``lru_cache`` on the grid topology."""
    key = (int(in_size), int(out_size), str(device))
    ent = _resize_tables.get(key)
    if ent is None:
        import numpy as np
        lib = _lib.load()
        ksize = int(lib.gnc_resize_bicubic_ksize(in_size, out_size))
        if ksize <= 0:
            raise ValueError(f"resize_bicubic: bad sizes {in_size} -> {out_size}")
        bounds = np.empty((out_size, 2), np.int32)
        kk = np.empty((out_size, ksize), np.int32)
        check(lib.gnc_resize_bicubic_coeffs(in_size, out_size, bounds.ctypes.data, kk.ctypes.data), "resize_bicubic_coeffs")
        if len(_resize_tables) >= 512:
            _resize_tables.clear()
        ent = _resize_tables[key] = (torch.from_numpy(bounds).to(device), torch.from_numpy(kk).to(device), ksize)
    return ent


def resize_bicubic(images: Tensor, out_h: int, out_w: Optional[int] = None) -> Tensor:
    """``PIL.Image.resize((out_w, out_h))`` (BICUBIC, Pillow's default for RGB) of ``uint8 [H, W, 3]`` or
    ``[B, H, W, 3]`` CUDA images, bit-identical to Pillow - the resize the reference's builders apply
    (utils/image_to_graph/image_to_graph_optimized.py:65-70).  Returns ``uint8 [(B,) out_h, out_w, 3]``."""
    _require_cuda(images)
    if images.dtype != torch.uint8 or images.dim() not in (3, 4) or images.shape[-1] != 3:
        raise ValueError(f"resize_bicubic expects uint8 [.., H, W, 3], got {images.dtype} {tuple(images.shape)}")
    out_w = out_h if out_w is None else out_w
    single = images.dim() == 3
    img = images.unsqueeze(0) if single else images
    if img.stride(3) != 1 or img.stride(2) != 3:
        img = img.contiguous()
    B, H, W, _ = img.shape
    dev = img.device
    dst = torch.empty(B, out_h, out_w, 3, dtype=torch.uint8, device=dev)
    bx = kx = by = ky = None
    ksx = ksy = 0
    if W != out_w:
        bx, kx, ksx = _resize_axis_tables(W, out_w, dev)
    if H != out_h:
        by, ky, ksy = _resize_axis_tables(H, out_h, dev)
    tmp = torch.empty(B, H, out_w, 3, dtype=torch.uint8, device=dev) if (bx is not None and by is not None) else None
    pitch = img.stride(1) if H > 1 else 3 * W
    istride = img.stride(0) if B > 1 else H * pitch
    nbytes = 3.0 * B * (H * W + out_h * out_w)
    check(_call("resize_bicubic", 0.0, nbytes, _lib.load().gnc_resize_bicubic_u8, img.data_ptr(), B, H, W, pitch, istride,
                out_h, out_w, _p(bx), _p(kx), ksx, _p(by), _p(ky), ksy, _p(tmp), dst.data_ptr(), _stream()), "resize_bicubic")
    return dst[0] if single else dst


def _ragged_plan(heights, widths, out_h: int, out_w: int):
    """Host half of ``resize_bicubic_ragged``, from the shapes alone: a ``gnc_resize_image`` record per image with its
    taps per axis (0 where the size is already the target), its table offsets and its first row of the horizontal
    pass's output.  Returns ``(records, table int32 elements, horizontal-pass rows, widest width changed)``; the
    caller fills ``src`` and ``pitch``."""
    import numpy as np
    h = np.asarray(heights, np.int64)
    w = np.asarray(widths, np.int64)

    def taps(size, out):                    # gnc_resize_bicubic_ksize: ceil(2 max(in / out, 1)) * 2 + 1
        return np.where(size != out, np.ceil(2.0 * np.maximum(size / out, 1.0)).astype(np.int64) * 2 + 1, 0)

    kx, ky = taps(w, out_w), taps(h, out_h)
    x_len = np.where(kx > 0, out_w * (2 + kx), 0)
    y_len = np.where(ky > 0, out_h * (2 + ky), 0)
    tab_x = np.cumsum(x_len + y_len) - (x_len + y_len)
    h_rows = np.where(kx > 0, h, 0)
    rec = np.zeros(len(h), np.dtype(_lib.GncResizeImage))
    rec["height"], rec["width"], rec["ksize_x"], rec["ksize_y"] = h, w, kx, ky
    rec["tab_x"], rec["tab_y"] = tab_x, tab_x + x_len
    rec["tmp_row"] = np.cumsum(h_rows) - h_rows
    max_w = int(w[kx > 0].max()) if (kx > 0).any() else 0
    return rec, int((x_len + y_len).sum()), int(h_rows.sum()), max_w


def resize_bicubic_ragged(images: Sequence[Tensor], out_h: int, out_w: Optional[int] = None) -> Tensor:
    """``PIL.Image.resize((out_w, out_h))`` of every image of a list of CUDA ``uint8 [H_i, W_i, 3]`` tensors of any
    sizes (strided views too) -> ``uint8 [n, out_h, out_w, 3]``, bit-identical to ``resize_bicubic`` of each image.
    Three launches whatever the number of shapes: the coefficient tables are computed on the device, and the image
    records reach it in one copy from pinned memory.  ``resize_bicubic`` stays the form for batches of one shape."""
    import numpy as np
    out_w = out_h if out_w is None else out_w
    if out_h <= 0 or out_w <= 0:
        raise ValueError(f"resize_bicubic_ragged: bad output size {out_h} x {out_w}")
    n = len(images)
    if n == 0:
        dev = torch.device("cuda", torch.cuda.current_device())
        return torch.empty(0, out_h, out_w, 3, dtype=torch.uint8, device=dev)
    _require_cuda(*images)
    dev = images[0].device
    srcs = []
    for t in images:
        if t.dtype != torch.uint8 or t.dim() != 3 or t.shape[2] != 3 or t.shape[0] == 0 or t.shape[1] == 0:
            raise ValueError(f"resize_bicubic_ragged expects uint8 [H, W, 3] images, got {t.dtype} {tuple(t.shape)}")
        if t.device != dev:
            raise ValueError(f"resize_bicubic_ragged: images on {t.device} and {dev}")
        if t.stride(2) != 1 or (t.shape[1] > 1 and t.stride(1) != 3):
            t = t.contiguous()
        srcs.append(t)
    rec, n_tables, h_rows, max_w = _ragged_plan([t.shape[0] for t in srcs], [t.shape[1] for t in srcs], out_h, out_w)
    rec["src"] = [t.data_ptr() for t in srcs]
    rec["pitch"] = [t.stride(0) if t.shape[0] > 1 else 3 * t.shape[1] for t in srcs]
    host = torch.empty(rec.nbytes, dtype=torch.uint8, pin_memory=True)
    host.numpy()[:] = rec.view(np.uint8)
    records = host.to(dev, non_blocking=True)       # the host allocator keeps `host` until this copy has run
    tables = torch.empty(max(n_tables, 1), dtype=torch.int32, device=dev)
    tmp = torch.empty(h_rows * 3 * out_w, dtype=torch.uint8, device=dev) if h_rows else None
    dst = torch.empty(n, out_h, out_w, 3, dtype=torch.uint8, device=dev)
    nbytes = 3.0 * (sum(t.shape[0] * t.shape[1] for t in srcs) + n * out_h * out_w)
    check(_call("resize_bicubic_ragged", 0.0, nbytes, _lib.load().gnc_resize_bicubic_ragged_u8, records.data_ptr(), n, out_h,
                out_w, h_rows, max_w, tables.data_ptr(), _p(tmp), dst.data_ptr(), _stream()), "resize_bicubic_ragged")
    return dst


class _ScatterSumFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src, rowptr, eid, idx32, n_rows):
        ctx.save_for_backward(idx32)
        return _agg_raw(rowptr, eid, src, n_rows)

    @staticmethod
    def backward(ctx, dout):
        (idx32,) = ctx.saved_tensors
        return _gather_raw(dout, idx32), None, None, None, None


def scatter_sum(src: Tensor, index: Tensor, dim: int = 0, dim_size: Optional[int] = None) -> Tensor:
    """Drop-in for the reference's module-level ``scatter_sum`` (models/GNN.py:3-21):
    rows of ``src`` summed into ``out[index]`` in ascending row order; new tensor;
    ``dim_size`` defaults to ``index.max() + 1`` (a host sync, as in the reference)."""
    if dim != 0:
        raise NotImplementedError("scatter_sum supports dim=0 only")
    _require_cuda(src, index)
    if src.dim() == 1:
        src = src.unsqueeze(-1)
    E = int(index.shape[0])
    if dim_size is None:
        dim_size = int(index.max().item()) + 1 if E > 0 else 0
    N = int(dim_size)
    dev = src.device
    if N == 0:
        return src.new_zeros((0, src.shape[1]))
    lib = _lib.load()
    key = index if index.dtype == torch.int64 else index.long()
    rowptr = torch.empty(N + 1, dtype=torch.int32, device=dev)
    eid = torch.empty(max(E, 1), dtype=torch.int32, device=dev)[:E]
    key32 = torch.empty(max(E, 1), dtype=torch.int32, device=dev)[:E]
    bad = torch.zeros(1, dtype=torch.int32, device=dev)
    work = _workspace(dev, int(lib.gnc_csr_workspace(N)), torch.int32)
    check(lib.gnc_csr_build(key.data_ptr(), key.stride(0) if E > 1 else 1, E, N, rowptr.data_ptr(), eid.data_ptr(),
                            key32.data_ptr(), work.data_ptr(), bad.data_ptr(), _stream()), "csr_build")
    if int(bad.item()) != 0:
        raise IndexError(f"scatter_sum: index out of range for dim_size {N}")
    return _ScatterSumFn.apply(src, rowptr, eid, key32, N)


# ----------------------------------------------------------------------------
# tensor-core engine (no autograd: used by the inference path)
# ----------------------------------------------------------------------------
def tc_linear(A: Tensor, W: Tensor, *, transpose_w: bool = False, bias: Optional[Tensor] = None,
              addend: Optional[Tensor] = None, gather0=None, gather1=None, relu: bool = False,
              gamma: Optional[Tensor] = None, beta: Optional[Tensor] = None, eps: float = 1e-5,
              residual: Optional[Tensor] = None, dot_w: Optional[Tensor] = None,
              dot_b: Optional[Tensor] = None, mask: Optional[Tensor] = None,
              out: Optional[Tensor] = None, ln_save=None) -> Tensor:
    """``epilogue(A @ W.T)`` on the tcgen05 3xTF32 engine (``A @ W`` with transpose_w).
    ``gather0`` / ``gather1`` are ``(rows [R, 128], idx int32 [M])`` pairs added row-wise as
    ``rows[idx[m]]``.  See include/gnc.h ``gnc_tc_epilogue_t`` for the epilogue algebra."""
    _require_cuda(A, W)
    A = _rows(A)
    M, K = A.shape
    N = W.shape[1] if transpose_w else W.shape[0]
    if W.dtype != torch.float32 or W.device != A.device or K != (W.shape[0] if transpose_w else W.shape[1]):
        raise RuntimeError(f"tc_linear: input width {K} / weight {tuple(W.shape)} {W.dtype} on {W.device} do not match")
    if bias is not None and (bias.numel() != N or bias.dtype != torch.float32 or bias.device != A.device):
        raise RuntimeError(f"tc_linear: bias must be a float32 vector of {N} elements on {A.device}")
    if W.stride(1) != 1:
        W = W.contiguous()
    epi = GncTcEpilogue()
    keep = []

    def rows(t):
        t = _rows(t)
        keep.append(t)
        return t

    if bias is not None:
        epi.bias = bias.data_ptr()
    if addend is not None:
        t = rows(addend)
        epi.addend, epi.ld_addend = t.data_ptr(), _ld(t)
    if gather0 is not None:
        t = rows(gather0[0])
        epi.gather0, epi.gather0_idx, epi.ld_gather0 = t.data_ptr(), gather0[1].data_ptr(), _ld(t)
    if gather1 is not None:
        t = rows(gather1[0])
        epi.gather1, epi.gather1_idx, epi.ld_gather1 = t.data_ptr(), gather1[1].data_ptr(), _ld(t)
    epi.relu = int(bool(relu))
    if gamma is not None:
        epi.gamma, epi.beta, epi.eps = gamma.data_ptr(), beta.data_ptr(), float(eps)
    res_rows = 0
    if residual is not None:
        if isinstance(residual, tuple):           # (table, idx int32 [M]): residual row = table[idx[m]]
            t = rows(residual[0])
            epi.residual, epi.ld_residual, epi.residual_idx = t.data_ptr(), _ld(t), residual[1].data_ptr()
            res_rows = t.shape[0]
        else:
            t = rows(residual)
            epi.residual, epi.ld_residual = t.data_ptr(), _ld(t)
            res_rows = M
    if mask is not None:
        t = rows(mask)
        epi.mask, epi.ld_mask = t.data_ptr(), _ld(t)
    if ln_save is not None:                       # (z [M, 128], mean [M], rstd [M]) outputs of the LayerNorm epilogue
        if gamma is None:
            raise ValueError("ln_save belongs to the LayerNorm epilogue (gamma / beta)")
        z_out, mean_out, rstd_out = ln_save
        epi.ln_z, epi.ld_ln_z = z_out.data_ptr(), _ld(z_out)
        epi.ln_mean, epi.ln_rstd = mean_out.data_ptr(), rstd_out.data_ptr()
    if dot_w is not None:
        dw = dot_w.reshape(-1)
        if dw.stride(0) != 1:
            dw = dw.contiguous()
        keep.append(dw)
        epi.dot_w = dw.data_ptr()
        epi.dot_b = None if dot_b is None else dot_b.data_ptr()
    n_out = 1 if dot_w is not None else N
    if out is None:
        out = torch.empty(M, n_out, dtype=torch.float32, device=A.device)
    # algorithmic HBM bytes: every operand row once (gathered tables count their own rows, not
    # one row per reference - re-references are expected to hit L2)
    nbytes = 4.0 * (M * K + M * n_out + N * K
                    + M * 128 * ((addend is not None) + (mask is not None) + (ln_save is not None)) + res_rows * 128
                    + (gather0[0].shape[0] * 128 + M if gather0 is not None else 0)
                    + (gather1[0].shape[0] * 128 + M if gather1 is not None else 0))
    check(_call("tc_linear", 2.0 * M * N * K, nbytes, _lib.load().gnc_tc_linear_f32, A.data_ptr(), _ld(A), M, K,
                W.data_ptr(), W.stride(0), N, int(transpose_w), ctypes.byref(epi), out.data_ptr(), _ld(out),
                _stream()), "tc_linear")
    return out


def tc_linear_multi(A: Tensor, weights: Sequence[Tensor], engine: str = "chain") -> list:
    """``[A @ W.T for W in weights]`` (2 or 3 width-128 weights, e.g. column slices of wider
    matrices) in one launch.  ``engine="chain"``: the chained kernel in multi mode (A stays in tensor
    memory for all products, fp16 two-piece operands); ``"tf32"``: the co-scheduled 3xTF32 launch
    whose CTAs share the A tiles through L2."""
    _require_cuda(A, *weights)
    A = _rows(A)
    M = A.shape[0]
    n = len(weights)
    Ws = [w if w.stride(1) == 1 else w.contiguous() for w in weights]
    outs = [torch.empty(M, 128, dtype=torch.float32, device=A.device) for _ in range(n)]
    wp = (ctypes.c_void_p * n)(*[w.data_ptr() for w in Ws])
    ld = (ctypes.c_int64 * n)(*[w.stride(0) for w in Ws])
    yp = (ctypes.c_void_p * n)(*[o.data_ptr() for o in outs])
    nbytes = 4.0 * 128 * (M + n * M + n * 128)
    if engine == "chain":
        check(_call("tc_mlp_chain", 2.0 * M * 128 * 128 * n, nbytes, _lib.load().gnc_tc_multi_chain_f32,
                    A.data_ptr(), _ld(A), M, n, wp, ld, None, yp, 128, _stream()), "tc_multi_chain")
    else:
        check(_call("tc_linear", 2.0 * M * 128 * 128 * n, nbytes, _lib.load().gnc_tc_linear_multi_f32,
                    A.data_ptr(), _ld(A), M, n, wp, ld, yp, 128, _stream()), "tc_linear_multi")
    return outs


def tc_mlp_chain(A: Optional[Tensor], layers: Sequence, *, gather0=None, gather1=None, gamma: Optional[Tensor] = None,
                 beta: Optional[Tensor] = None, eps: float = 1e-5, residual=None, dot_w: Optional[Tensor] = None,
                 dot_b: Optional[Tensor] = None, out: Optional[Tensor] = None, pre=None, operand2=None,
                 narrow=None, stash=None, agg=None, edge_slots: int = 0, paired: bool = False) -> Tensor:
    """Two or three chained ``Linear(128, 128)`` layers in one launch (csrc/tc_chain.cu), ReLU after
    all but the last, hidden activations kept on chip.  ``layers`` is ``[(W, bias), ...]``;
    ``gather0`` / ``gather1`` are ``(rows, idx int32 [M] | None)`` pre-activation addends of the first
    layer (``idx=None``: row m); the tail is ``LayerNorm(gamma, beta) + residual`` (``residual`` a
    tensor or ``(table, idx)``) or the decoder's ``relu(.) . dot_w + dot_b``.
    ``narrow=(Wn [128, k<=8], bn)``: ``A`` has k columns and the first operand is ``relu(A @ Wn.T + bn)`` (the
    encoders' first layer folded into the launch).  ``operand2=(A2, W_A2)`` adds ``A2 @ W_A2.T`` to the first layer (two-operand contraction, no addend tensor).
    ``A=None`` with ``pre=(table, idx int32 [M], bias)`` is the pre-stage form: the first operand is
    ``relu(table[idx] + gather0 + gather1 + bias)`` and ``layers`` are the two layers after it.
    ``agg=(rowptr int32 [M + 1], eid int32)`` with ``operand2``: ``A`` is the ``[E, 128]`` edge table and the first operand's
    row ``m`` is the ordered sum of ``A[eid[k]]``, ``k`` in ``[rowptr[m], rowptr[m + 1])`` - at most two entries per row
    (``scatter_sum`` folded into the launch; the caller has checked the in-degrees).
    ``edge_slots`` (edge processor forms; ``gather0`` / ``gather1`` indexed by ``GraphIndex.pair_slots``): 1 - the rows are
    paired destination slots and a slot whose ``gather0`` index is negative gets the row +0.0; 2 - and the result is the
    ``[M / 2, 128]`` per-node sum ``(0 + y[2v]) + y[2v + 1]`` instead of the slot rows.
    ``paired=True`` with ``operand2``: ``A`` is the ``[2 M, 128]`` slot table and the first operand's row ``m`` is
    ``(0 + A[2m]) + A[2m + 1]``.
    ``stash=(a1, a2, z, mean, rstd)`` (training forward of a block's edge / node MLP: 3 layers, addends, LayerNorm, residual
    by row): the launch also writes the hidden ReLU outputs ``a1``, ``a2``, the LayerNorm input ``z`` (``[M, 128]`` each) and
    the row statistics ``mean``, ``rstd`` (``[M]``) - what the backward pass of the MLP reads.
    See include/gnc.h ``gnc_tc_chain_t``."""
    ch = GncTcChain()
    keep = []
    if A is None:
        tab, tidx, tbias = pre
        tab = _rows(tab)
        keep.append(tab)
        M = tidx.shape[0]
        ch.gather2, ch.gather2_idx, ch.ld_gather2 = tab.data_ptr(), tidx.data_ptr(), _ld(tab)
        ch.pre_bias = None if tbias is None else tbias.data_ptr()
        a_ptr, a_ld, dev = None, 0, tab.device
    else:
        _require_cuda(A)
        A = _rows(A)
        M = A.shape[0]
        if agg is not None:
            if operand2 is None:
                raise ValueError("tc_mlp_chain: agg goes with operand2 (the node processor's two-operand form)")
            rp, ei = agg
            if rp.dtype != torch.int32 or ei.dtype != torch.int32 or rp.device != A.device or ei.device != A.device:
                raise ValueError("tc_mlp_chain: agg = (rowptr, eid) int32 tensors on the operands' device")
            M = rp.numel() - 1
            keep += [rp, ei]
            ch.agg_rowptr, ch.agg_eid = rp.data_ptr(), ei.data_ptr()
        if paired:
            if operand2 is None or agg is not None or M % 2 != 0:
                raise ValueError("tc_mlp_chain: paired goes with operand2, without agg, on an even number of slot rows")
            M //= 2
            ch.paired_operand = 1
        a_ptr, a_ld, dev = A.data_ptr(), _ld(A), A.device
        if narrow is not None:
            Wn, bn = narrow
            if Wn.stride(1) != 1:
                Wn = Wn.contiguous()
            keep.append(Wn)
            ch.narrow_W, ch.ld_narrow_W, ch.narrow_k = Wn.data_ptr(), Wn.stride(0), Wn.shape[1]
            ch.narrow_b = None if bn is None else bn.data_ptr()
    ch.nlayers = len(layers)
    for l, (W, b) in enumerate(layers):
        _require_cuda(W)
        if tuple(W.shape) != (128, 128) or W.dtype != torch.float32 or (b is not None and (b.numel() != 128 or b.dtype != torch.float32)):
            raise RuntimeError(f"tc_mlp_chain: layer {l} must be a float32 [128, 128] weight with a 128-element bias, "
                               f"got {tuple(W.shape)} {W.dtype}")
        if W.stride(1) != 1:
            W = W.contiguous()
        keep.append(W)
        ch.W[l], ch.ldw[l] = W.data_ptr(), W.stride(0)
        ch.bias[l] = None if b is None else b.data_ptr()
    nbytes = 4.0 * (((A.shape[0] if (agg is not None or paired) else M) * (A.shape[1] if narrow is not None else 128) if A is not None else 0)
                    + len(layers) * 128 * 128 + (2 * M + 1 if agg is not None else 0))
    if operand2 is not None:
        A2, W2 = operand2
        A2 = _rows(A2)
        if W2.stride(1) != 1:
            W2 = W2.contiguous()
        keep += [A2, W2]
        ch.operand2, ch.ld_operand2, ch.W_operand2, ch.ldw_operand2 = A2.data_ptr(), _ld(A2), W2.data_ptr(), W2.stride(0)
        nbytes += 4.0 * 128 * (M + 128)

    def rows(t):
        t = _rows(t)
        keep.append(t)
        return t

    for name, g in (("gather0", gather0), ("gather1", gather1)):
        if g is None:
            continue
        t = rows(g[0])
        setattr(ch, name, t.data_ptr())
        setattr(ch, "ld_" + name, _ld(t))
        if g[1] is not None:
            setattr(ch, name + "_idx", g[1].data_ptr())
        nbytes += 4.0 * (t.shape[0] * 128 + (M if g[1] is not None else 0))
    if gamma is not None:
        ch.gamma, ch.beta = gamma.data_ptr(), beta.data_ptr()
    ch.eps = float(eps)
    if residual is not None:
        if isinstance(residual, tuple):
            t = rows(residual[0])
            ch.residual, ch.ld_residual, ch.residual_idx = t.data_ptr(), _ld(t), residual[1].data_ptr()
        else:
            t = rows(residual)
            ch.residual, ch.ld_residual = t.data_ptr(), _ld(t)
        nbytes += 4.0 * t.shape[0] * 128
    n_out, m_out = 128, M
    if edge_slots:
        if edge_slots not in (1, 2) or (edge_slots == 2 and M % 2 != 0):
            raise ValueError("tc_mlp_chain: edge_slots is 1, or 2 on an even number of slot rows")
        ch.edge_slots = int(edge_slots)
        if edge_slots == 2:
            m_out = M // 2
    if dot_w is not None:
        dw = dot_w.reshape(-1)
        if dw.stride(0) != 1:
            dw = dw.contiguous()
        keep.append(dw)
        ch.dot_w = dw.data_ptr()
        ch.dot_b = None if dot_b is None else dot_b.data_ptr()
        n_out = 1
    if out is None:
        out = torch.empty(m_out, n_out, dtype=torch.float32, device=dev)
    nbytes += 4.0 * m_out * n_out
    if stash is not None:
        a1s, a2s, zs, means, rstds = stash
        for t in (a1s, a2s, zs):
            if t.dtype != torch.float32 or t.device != dev or tuple(t.shape) != (M, 128) or t.stride(1) != 1 or t.stride(0) != a1s.stride(0):
                raise ValueError("tc_mlp_chain: stash a1 / a2 / z must be float32 [M, 128] row sets of one pitch on the operands' device")
        for t in (means, rstds):
            if t.dtype != torch.float32 or t.device != dev or t.numel() != M or not t.is_contiguous():
                raise ValueError("tc_mlp_chain: stash mean / rstd must be contiguous float32 [M]")
        ch.stash_a1, ch.stash_a2, ch.stash_z, ch.ld_stash = a1s.data_ptr(), a2s.data_ptr(), zs.data_ptr(), a1s.stride(0)
        ch.stash_mean, ch.stash_rstd = means.data_ptr(), rstds.data_ptr()
        nbytes += 4.0 * M * (3 * 128 + 2)
    check(_call("tc_mlp_chain", 2.0 * M * 128 * 128 * (len(layers) + (operand2 is not None)), nbytes,
                _lib.load().gnc_tc_mlp_chain_f32,
                a_ptr, a_ld, M, ctypes.byref(ch), out.data_ptr(), _ld(out), _stream()), "tc_mlp_chain")
    return out


class _TcLinearFn(torch.autograd.Function):
    """``act(A @ W.T + b + addend + P[src] + Q[dst])`` on the tensor-core engine, with its
    backward: weight + bias gradients in one tcgen05 pass (gnc_tc_wgrad_f32), data gradient on
    the tensor-core engine (B = W^T), gathered addends' gradients as ordered CSR segmented sums.

    ReLU backward is fused along MLP chains instead of being a pass of its own:
      * ``mask_input``  - ``A`` is the ReLU output of the layer before; the data gradient is
        multiplied by ``(A > 0)`` in the GEMM epilogue, i.e. it is already the gradient with
        respect to that layer's pre-activation;
      * ``premasked``   - this layer's own ReLU mask has been applied to the incoming gradient by
        its (single) consumer, which was built with ``mask_input``; nothing is left to do.
    Masking twice would also be correct (the mask is idempotent); the flags only remove passes."""

    @staticmethod
    def forward(ctx, A, W, b, relu, addend, P, Q, gmeta, mask_input, premasked):
        A = _rows(A)
        Wc = W if W.stride(1) == 1 else W.contiguous()
        g0 = (P, gmeta[0]) if P is not None else None
        g1 = (Q, gmeta[2]) if Q is not None else None
        Y = tc_linear(A, Wc, bias=b, relu=relu, addend=addend, gather0=g0, gather1=g1)
        ctx.relu, ctx.gmeta, ctx.has_bias = bool(relu), gmeta, b is not None
        ctx.mask_input, ctx.premasked = bool(mask_input), bool(premasked)
        ctx.save_for_backward(A, Wc, Y if (relu and not premasked) else None)
        return Y

    @staticmethod
    def backward(ctx, dY):
        A, Wc, Y = ctx.saved_tensors
        lib = _lib.load()
        dev = dY.device
        M, N = A.shape[0], Wc.shape[0]
        dY = _rows(dY)
        need = ctx.needs_input_grad          # (A, W, b, relu, addend, P, Q, gmeta, mask_input, premasked)
        need_b = need[2] and ctx.has_bias
        dZ = dY
        if ctx.relu and not ctx.premasked:
            dZ = torch.empty(M, N, dtype=torch.float32, device=dev)
            ws_n = int(lib.gnc_colsum_workspace(M, N))
            ws = _workspace(dev, ws_n)
            check(_call("relu_bwd_colsum", 0.0, 4.0 * M * N * 3, lib.gnc_relu_bwd_colsum_f32,
                        dY.data_ptr(), _ld(dY), Y.data_ptr(), _ld(Y), M, N, dZ.data_ptr(), _ld(dZ), None, 0,
                        ws.data_ptr(), ws_n, _stream()), "relu_bwd_colsum")
        dW = db = None
        if need[1] and need_b:
            dW, db = tc_wgrad(dZ, A, want_db=True)
        elif need[1]:
            dW = tc_wgrad(dZ, A)
        elif need_b:
            db = torch.empty(N, dtype=torch.float32, device=dev)
            ws_n = int(lib.gnc_colsum_workspace(M, N))
            ws = _workspace(dev, ws_n)
            check(_call("relu_bwd_colsum", 0.0, 4.0 * M * N, lib.gnc_relu_bwd_colsum_f32, dZ.data_ptr(), _ld(dZ), None, 0,
                        M, N, None, 0, db.data_ptr(), 0, ws.data_ptr(), ws_n, _stream()), "relu_bwd_colsum")
        dA = None
        if need[0]:
            dA = tc_linear(dZ, Wc, transpose_w=True, mask=A if ctx.mask_input else None)
        daddend = dZ if need[4] else None
        dP = dQ = None
        if need[5]:
            _, src_csr, _, _, n_nodes = ctx.gmeta
            dP = _agg_raw(src_csr[0], src_csr[1], dZ, n_nodes)
        if need[6]:
            _, _, _, dst_csr, n_nodes = ctx.gmeta
            dQ = _agg_raw(dst_csr[0], dst_csr[1], dZ, n_nodes)
        return dA, dW, db, None, daddend, dP, dQ, None, None, None


def tc_linear_autograd(A: Tensor, W: Tensor, b: Optional[Tensor] = None, relu: bool = False,
                       addend: Optional[Tensor] = None, P: Optional[Tensor] = None, Q: Optional[Tensor] = None,
                       graph: Optional[GraphIndex] = None, mask_input: bool = False,
                       premasked: bool = False) -> Tensor:
    """Differentiable tensor-core linear layer (width 128).  ``P`` / ``Q`` are node tables added
    as ``P[graph.src]`` / ``Q[graph.dst]`` (the edge processor's first layer, see GraphNet).
    ``mask_input`` / ``premasked``: ReLU-backward fusion flags, see ``_TcLinearFn``."""
    gmeta = None
    if P is not None or Q is not None:
        gmeta = (graph.src, (graph.src_rowptr, graph.src_eid), graph.dst, (graph.dst_rowptr, graph.dst_eid),
                 graph.num_nodes)
    return _TcLinearFn.apply(A, W, b, relu, addend, P, Q, gmeta, mask_input, premasked)


def tc_wgrad(dZ: Tensor, X: Tensor, out: Optional[Tensor] = None, accumulate: bool = False,
             want_db: bool = False):
    """``dZ.T @ X`` for ``[M, 128]`` operands on the tensor-core engine (weight gradient);
    with ``want_db`` also the column sums of ``dZ`` (bias gradient) from the same pass."""
    _require_cuda(dZ, X)
    dZ, X = _rows(dZ), _rows(X)
    M = dZ.shape[0]
    lib = _lib.load()
    if out is None:
        out = torch.empty(dZ.shape[1], X.shape[1], dtype=torch.float32, device=dZ.device)
        accumulate = False
    db = torch.empty(dZ.shape[1], dtype=torch.float32, device=dZ.device) if want_db else None
    ws_n = int(lib.gnc_tc_wgrad_workspace(M))
    ws = _workspace(dZ.device, ws_n)
    check(_call("tc_wgrad", 2.0 * M * dZ.shape[1] * X.shape[1], 4.0 * M * (dZ.shape[1] + X.shape[1]),
                lib.gnc_tc_wgrad_f32, dZ.data_ptr(), _ld(dZ), X.data_ptr(), _ld(X), M, dZ.shape[1], X.shape[1],
                out.data_ptr(), _ld(out), int(accumulate), _p(db), ws.data_ptr(), ws_n, _stream()), "tc_wgrad")
    return (out, db) if want_db else out


class DeferredBwdReduce:
    """Collects the weight / bias gradient reductions of the fused backward-layer launches of one backward pass and
    finishes them with ONE launch (``gnc_tc_bwd_reduce_batch_f32``) instead of one small launch per layer.  While
    active (``with ops.DeferredBwdReduce():``), ``tc_bwd_layer`` leaves every layer's per-CTA partial sums in a
    workspace of its own; ``dW`` / ``db`` tensors it returns are valid after the ``with`` block (or ``flush()``)."""

    active: Optional["DeferredBwdReduce"] = None

    def __init__(self):
        self.items = []          # (workspace, parts, dW, db, accumulate)

    def __enter__(self):
        self._prev, DeferredBwdReduce.active = DeferredBwdReduce.active, self
        return self

    def __exit__(self, exc_type, exc, tb):
        DeferredBwdReduce.active = self._prev
        if exc_type is None:
            self.flush()
        self.items = []
        return False

    def flush(self) -> None:
        if not self.items:
            return
        arr = (_lib.GncBwdReduceItem * len(self.items))()
        for a, (ws, parts, dW, db, acc) in zip(arr, self.items):
            a.work, a.dW, a.db = ws.data_ptr(), _p(dW), _p(db)
            a.lddw, a.parts, a.accumulate = (dW.stride(0) if dW is not None else 0), parts, int(acc)
        n = len(self.items)
        check(_call("tc_bwd_reduce_batch", 0.0, sum(4.0 * it[1] * (128 * 128 + 128) for it in self.items),
                    _lib.load().gnc_tc_bwd_reduce_batch_f32, arr, n, _stream()), "tc_bwd_reduce_batch")
        self.items = []


def tc_bwd_layer(dZ: Tensor, X: Tensor, W: Tensor, *, mask: bool = False, addend: Optional[Tensor] = None,
                 dW_out: Optional[Tensor] = None, accumulate: bool = False, want_db: bool = False,
                 db_out: Optional[Tensor] = None, want_dW: bool = True):
    """Backward of ``y = x @ W.T (+ b)`` for ``[M, 128]`` operands in ONE pass over ``dZ`` and ``X`` (csrc/tc_bwd.cu):
    returns ``(dX, dW, db)`` with ``dX = dZ @ W`` (``* (X > 0)`` with ``mask``, ``+ addend``), ``dW = dZ.T @ X``
    (written into ``dW_out`` when given, added to it with ``accumulate``; ``accumulate`` also applies to ``db_out``)
    and ``db`` = column sums of ``dZ`` (``None`` unless asked for)."""
    _require_cuda(dZ, X, W)
    dZ, X = _rows(dZ), _rows(X)
    M = dZ.shape[0]
    if dZ.shape[1] != 128 or X.shape != dZ.shape or tuple(W.shape) != (128, 128):
        raise ValueError(f"tc_bwd_layer: width-128 operands only, got dZ {tuple(dZ.shape)}, X {tuple(X.shape)}, W {tuple(W.shape)}")
    if W.dtype != torch.float32 or W.device != dZ.device or X.device != dZ.device:
        raise ValueError("tc_bwd_layer: W / X must be float32 tensors on dZ's device")
    if W.stride(1) != 1:
        W = W.contiguous()
    lib = _lib.load()
    dev = dZ.device
    dX = torch.empty(M, 128, dtype=torch.float32, device=dev)
    ad = None
    if addend is not None:
        ad = _rows(addend)
        if ad.shape != dZ.shape:
            raise ValueError("tc_bwd_layer: addend must have dZ's shape")
    dW = None
    if want_dW:
        if dW_out is None:
            if accumulate:
                raise ValueError("tc_bwd_layer: accumulate needs dW_out")
            dW = torch.empty(128, 128, dtype=torch.float32, device=dev)
        else:
            dW = dW_out
            if tuple(dW.shape) != (128, 128) or dW.stride(1) != 1 or dW.dtype != torch.float32:
                raise ValueError("tc_bwd_layer: dW_out must be a float32 [128, 128] view with unit column stride")
    db = None
    if want_db:
        if db_out is None and accumulate:
            raise ValueError("tc_bwd_layer: accumulate with want_db needs db_out")
        db = db_out if db_out is not None else torch.empty(128, dtype=torch.float32, device=dev)
    ws_n = int(lib.gnc_tc_bwd_layer_workspace())
    defer = DeferredBwdReduce.active if (dW is not None or db is not None) else None
    if defer is not None:
        # the partial sums stay in a workspace of this layer's own until the pass's single reduction launch
        parts = int(lib.gnc_tc_bwd_layer_parts(M))
        ws = torch.empty(parts * (128 * 128 + 128), dtype=torch.float32, device=dev)
        defer.items.append((ws, parts, dW, db, bool(accumulate)))
        k_dW, k_db = None, None
    else:
        ws = _workspace(dev, ws_n)
        k_dW, k_db = dW, db
    check(_call("tc_bwd_layer", 4.0 * M * 128 * 128, 4.0 * 128 * M * (3 + (ad is not None)),
                lib.gnc_tc_bwd_layer_f32, dZ.data_ptr(), _ld(dZ), X.data_ptr(), _ld(X), M, W.data_ptr(), W.stride(0),
                int(bool(mask)), _p(ad), _ld(ad) if ad is not None else 0, dX.data_ptr(), _ld(dX),
                _p(k_dW), dW.stride(0) if dW is not None else 0, _p(k_db), int(bool(accumulate)), ws.data_ptr(),
                ws.numel(), _stream()), "tc_bwd_layer")
    return dX, dW, db


def dot_tail_fwd(X: Tensor, w: Tensor, b: Optional[Tensor]) -> Tensor:
    """``X @ w.T + b`` for a one-row weight ``w [1, D]`` (the decoder's ``Linear(128, 1)``) as a row dot product: ``[M, 1]``."""
    _require_cuda(X, w)
    X = _rows(X)
    M, D = X.shape
    wv = w.reshape(-1)
    if wv.numel() != D or wv.dtype != torch.float32 or (b is not None and b.numel() != 1):
        raise RuntimeError(f"dot_tail: weight {tuple(w.shape)} does not match input width {D}")
    if wv.stride(0) != 1:
        wv = wv.contiguous()
    y = torch.empty(M, 1, dtype=torch.float32, device=X.device)
    check(_call("dot_tail_fwd", 2.0 * M * D, 4.0 * M * (D + 1), _lib.load().gnc_dot_tail_fwd_f32, X.data_ptr(), _ld(X), M, D,
                wv.data_ptr(), _p(b), y.data_ptr(), _stream()), "dot_tail_fwd")
    return y


def dot_tail_bwd(X: Tensor, w: Tensor, dy: Tensor, relu_mask: bool = False, want_dX: bool = True,
                 dw_out: Optional[Tensor] = None, db_out: Optional[Tensor] = None):
    """Backward of ``dot_tail_fwd`` in one pass over ``X``: ``(dX, dw [1, D], db [1])`` with ``dX = dy * w``
    (``* (X > 0)`` with ``relu_mask``: then it is the pre-activation gradient of the ReLU that produced ``X``).
    With ``dw_out`` / ``db_out`` (both or neither) the parameter gradients are ADDED to those tensors."""
    _require_cuda(X, w, dy)
    X = _rows(X)
    M, D = X.shape
    wv = w.reshape(-1)
    if wv.stride(0) != 1:
        wv = wv.contiguous()
    g = dy.reshape(-1)
    if g.dtype != torch.float32 or g.stride(0) != 1:
        g = g.float().contiguous()
    if g.numel() != M or wv.numel() != D:
        raise RuntimeError("dot_tail_bwd: shapes do not match")
    lib = _lib.load()
    dev = X.device
    dX = torch.empty(M, D, dtype=torch.float32, device=dev) if want_dX else None
    acc = dw_out is not None
    if acc and (db_out is None or dw_out.numel() != D or not dw_out.is_contiguous() or db_out.numel() != 1):
        raise ValueError("dot_tail_bwd: dw_out [1, D] and db_out [1] come together, contiguous")
    dw = dw_out if acc else torch.empty(1, D, dtype=torch.float32, device=dev)
    db = db_out if acc else torch.empty(1, dtype=torch.float32, device=dev)
    ws_n = int(lib.gnc_dot_tail_bwd_workspace(M, D))
    ws = _workspace(dev, ws_n)
    check(_call("dot_tail_bwd", 4.0 * M * D, 4.0 * M * D * (2 if want_dX else 1), lib.gnc_dot_tail_bwd_f32, X.data_ptr(),
                _ld(X), M, D, wv.data_ptr(), g.data_ptr(), int(bool(relu_mask)), _p(dX), _ld(dX) if dX is not None else 0,
                dw.data_ptr(), db.data_ptr(), int(acc), ws.data_ptr(), ws_n, _stream()), "dot_tail_bwd")
    return dX, dw, db


class _CrossEntropyFn(torch.autograd.Function):
    """``scale * sum_b CE(logits[b], labels[b])`` (reference: nn.CrossEntropyLoss, utils/train_model.py:10, 38) with its
    gradient computed by the same launch."""

    @staticmethod
    def forward(ctx, logits, labels, scale, total):
        lg = _rows(logits)
        B, C = lg.shape
        lab = labels.reshape(-1)
        if lab.dtype != torch.int64 or lab.device != lg.device or lab.numel() != B:
            raise RuntimeError(f"cross_entropy: labels must be {B} int64 values on {lg.device}")
        if not lab.is_contiguous():
            lab = lab.contiguous()
        loss = torch.empty(1, dtype=torch.float32, device=lg.device)
        need = ctx.needs_input_grad[0]
        dl = torch.empty(B, C, dtype=torch.float32, device=lg.device) if need else None
        lib = _lib.load()
        check(_call("cross_entropy", 0.0, 8.0 * B * C, lib.gnc_cross_entropy_f32, lg.data_ptr(), _ld(lg), lab.data_ptr(), B, C,
                    float(scale), loss.data_ptr(), _p(total), _p(dl), C, None, _stream()), "cross_entropy")
        ctx.dl, ctx.shape = dl, logits.shape
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g):
        dl = ctx.dl
        ctx.dl = None
        # the upstream gradient of a loss is the scalar 1 in every use here; a different one scales the stored gradient
        return dl.reshape(ctx.shape) * g if dl is not None else None, None, None, None


def cross_entropy(logits: Tensor, labels: Tensor, scale: float = 1.0, total: Optional[Tensor] = None) -> Tensor:
    """``scale * sum_b CE(logits[b], labels[b])`` for ``[B, C]`` logits (``[C]`` = one graph) and int64 labels; with
    ``total`` (a 1-element fp32 device tensor) the value is also added to it."""
    _require_cuda(logits, labels)
    if logits.dim() == 1:
        logits = logits.reshape(1, -1)
    return _CrossEntropyFn.apply(logits, labels, float(scale), total)


def adam_step(param: Tensor, grad: Tensor, exp_avg: Tensor, exp_avg_sq: Tensor, step: int, lr: float = 1e-3,
              betas=(0.9, 0.999), eps: float = 1e-8, grad_scale: float = 1.0) -> None:
    """In-place Adam update of flat fp32 buffers (torch.optim.Adam's rule; ``step`` is the 1-based step count)."""
    _require_cuda(param, grad, exp_avg, exp_avg_sq)
    n = param.numel()
    for t in (param, grad, exp_avg, exp_avg_sq):
        if t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != n:
            raise RuntimeError("adam_step: flat contiguous fp32 buffers of equal length")
    check(_call("adam_step", 0.0, 28.0 * n, _lib.load().gnc_adam_step_f32, param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(),
                exp_avg_sq.data_ptr(), n, float(lr), float(betas[0]), float(betas[1]), float(eps), int(step), float(grad_scale),
                _stream()), "adam_step")


def zero_(buf: Tensor) -> None:
    """``buf[:] = 0`` for a contiguous fp32 device tensor (cudaMemsetAsync on the current stream)."""
    _require_cuda(buf)
    if buf.dtype != torch.float32 or not buf.is_contiguous():
        raise RuntimeError("zero_: contiguous fp32 tensor")
    check(_lib.load().gnc_zero_f32(buf.data_ptr(), buf.numel(), _stream()), "zero")


class _SegmentReadoutFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y, node_ptr, num_nodes):
        yv = y.reshape(-1)
        if yv.dtype != torch.float32 or not yv.is_contiguous():
            yv = yv.float().contiguous()
        B = int(node_ptr.shape[0]) - 1
        out = torch.empty(B, num_nodes, dtype=torch.float32, device=y.device)
        check(_call("segment_readout", 0.0, 4.0 * (yv.numel() + B * num_nodes), _lib.load().gnc_segment_readout_f32,
                    yv.data_ptr(), node_ptr.data_ptr(), B, int(num_nodes), out.data_ptr(), _stream()), "segment_readout")
        ctx.node_ptr, ctx.num_nodes, ctx.shape = node_ptr, int(num_nodes), y.shape
        return out

    @staticmethod
    def backward(ctx, dout):
        dout = _rows(dout)
        if _ld(dout) != ctx.num_nodes:
            dout = dout.contiguous()
        n_total = 1
        for d in ctx.shape:
            n_total *= d
        dy = torch.empty(n_total, dtype=torch.float32, device=dout.device)
        B = int(ctx.node_ptr.shape[0]) - 1
        check(_call("segment_readout_bwd", 0.0, 4.0 * (n_total + B * ctx.num_nodes), _lib.load().gnc_segment_readout_bwd_f32,
                    dout.data_ptr(), ctx.node_ptr.data_ptr(), B, ctx.num_nodes, dy.data_ptr(), _stream()), "segment_readout_bwd")
        return dy.reshape(ctx.shape), None, None


def segment_readout(y: Tensor, node_ptr: Tensor, num_nodes: int) -> Tensor:
    """Node outputs ``y [sum n_b, 1]`` of a batch of graphs with different node counts -> the dense ``[B, num_nodes]``
    input of the classifier head: graph ``b`` contributes its first ``min(n_b, num_nodes)`` outputs, missing entries are
    zero (SURVEY.md Q7: the reference's flatten, models/GNN.py:339, needs ``n_b == num_nodes`` and crashes otherwise)."""
    _require_cuda(y, node_ptr)
    if node_ptr.dtype != torch.int32 or node_ptr.dim() != 1 or node_ptr.shape[0] < 1:
        raise ValueError("segment_readout: node_ptr must be int32 [B + 1]")
    if y.numel() % max(int(y.shape[0]), 1) != 0 or y.numel() != y.shape[0]:
        raise ValueError("segment_readout: one output channel per node (out_channels = 1)")
    return _SegmentReadoutFn.apply(y, node_ptr.contiguous(), int(num_nodes))
