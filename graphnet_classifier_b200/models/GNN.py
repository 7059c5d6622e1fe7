"""GraphNet / CombinedModel with the reference's public surface (reference
models/GNN.py), running on libgnc kernels.

Same class names, constructor kwargs, forward signatures, attribute names and
``state_dict`` keys as the reference (76 tensors for the shipped configuration:
``graph_net.{node,edge}_encoder.model.*``, ``graph_net.graph_processor.blocks.k.
{edge_model.edge_processor,node_model.node_processor}.model.*``,
``graph_net.node_decoder.model.*``, ``classifier.fc{1,2,3}.*``), so checkpoints load
both ways.  What differs is underneath:

* the ``x[row]`` / ``x[col]`` gathers and both ``torch.cat`` calls are never
  materialised - the first Linear of each processor reads its operand through
  gathered column segments (include/gnc.h, ``gnc_seg_t``);
* ``scatter_sum`` is an ordered CSR segmented sum (bit-identical to the CPU
  reference's ``index_add_`` order);
* ``torch_geometric.nn.MetaLayer`` (un-vendored, no arithmetic) is replaced by the
  small ``MetaLayer`` below with the same attribute names;
* block-diagonal batches are accepted: ``x`` may hold ``B * num_nodes`` rows, logits
  come back ``[B, classes]`` (``[classes]`` for one graph, as the reference returns).
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn as nn
from torch import Tensor

from .. import ops, tc_train
from ..ops import GraphIndex, scatter_sum  # noqa: F401  (re-exported: reference module-level name)
from .MLP import MLP


class EdgeProcessor(nn.Module):
    """e' = MLP(cat[x_src, x_dst, e]) + e   (reference models/GNN.py:31-64)."""

    def __init__(self, in_dim_node: int, in_dim_edge: int, hidden_dim: int = 128, hidden_layers: int = 2,
                 activation: str = "ReLU", initializer: None | str = None, norm_type: None | str = "LayerNorm"):
        super().__init__()
        self.edge_processor = MLP(2 * in_dim_node + in_dim_edge, in_dim_edge, hidden_dim, hidden_layers,
                                  activation, initializer, norm_type)

    def forward(self, src, dest, edge_attr, u=None, batch=None):
        """MetaLayer calling convention: ``src`` / ``dest`` are already-gathered rows."""
        return self.edge_processor.forward_segments([src, dest, edge_attr], residual=edge_attr)

    def forward_graph(self, x: Tensor, graph: GraphIndex, edge_attr: Tensor) -> Tensor:
        """Same result from the un-gathered node latents: the gathers ride inside the
        first GEMM's operand loads; their backward is the CSR segmented sum."""
        gathers = [
            (graph.src, (graph.src_rowptr, graph.src_eid), graph.num_nodes),
            (graph.dst, (graph.dst_rowptr, graph.dst_eid), graph.num_nodes),
            None,
        ]
        return self.edge_processor.forward_segments([x, x, edge_attr], gathers=gathers, residual=edge_attr)


class NodeProcessor(nn.Module):
    """x' = MLP(cat[x, scatter_sum(e, col)]) + x   (reference models/GNN.py:69-104)."""

    def __init__(self, in_dim_node: int, in_dim_edge: int, hidden_dim: int = 128, hidden_layers: int = 2,
                 activation: str = "ReLU", initializer: None | str = None, norm_type: None | str = "LayerNorm"):
        super().__init__()
        self.node_processor = MLP(in_dim_node + in_dim_edge, in_dim_node, hidden_dim, hidden_layers,
                                  activation, initializer, norm_type)

    def forward(self, x: Tensor, edge_index: Tensor, edge_attr: Tensor, u=None, batch=None):
        return self.forward_graph(x, ops.graph_of(edge_index, x.size(0)), edge_attr)

    def forward_graph(self, x: Tensor, graph: GraphIndex, edge_attr: Tensor) -> Tensor:
        agg = ops.aggregate(edge_attr, graph)            # dim_size = N (SURVEY.md Q1)
        return self.node_processor.forward_segments([x, agg], residual=x)


class MetaLayer(nn.Module):
    """Stand-in for ``torch_geometric.nn.MetaLayer`` (reference models/GNN.py:24, 146):
    edge model on (x[row], x[col], edge_attr), then node model; no global model."""

    def __init__(self, edge_model=None, node_model=None, global_model=None):
        super().__init__()
        self.edge_model = edge_model
        self.node_model = node_model
        self.global_model = global_model

    def forward(self, x, edge_index, edge_attr=None, u=None, batch=None):
        graph = edge_index if isinstance(edge_index, GraphIndex) else ops.graph_of(edge_index, x.size(0))
        if self.edge_model is not None:
            if hasattr(self.edge_model, "forward_graph"):
                edge_attr = self.edge_model.forward_graph(x, graph, edge_attr)
            else:
                src = ops.gather_rows(x, graph.src, graph.src_rowptr, graph.src_eid)
                dst = ops.gather_rows(x, graph.dst, graph.dst_rowptr, graph.dst_eid)
                edge_attr = self.edge_model(src, dst, edge_attr, u, batch)
        if self.node_model is not None:
            if hasattr(self.node_model, "forward_graph"):
                x = self.node_model.forward_graph(x, graph, edge_attr)
            else:
                x = self.node_model(x, edge_index, edge_attr, u, batch)
        if self.global_model is not None:
            u = self.global_model(x, edge_index, edge_attr, u, batch)
        return x, edge_attr, u


def build_GN_block(in_dim_node: int, in_dim_edge: int, hidden_dim_node: int = 128, hidden_dim_edge: int = 128,
                   hidden_layers_node: int = 2, hidden_layers_edge: int = 2, activation: str = "ReLU",
                   initializer: None | str = None, norm_type: None | str = "LayerNorm"):
    """One message-passing block (reference models/GNN.py:110-165)."""
    edge_model = EdgeProcessor(in_dim_node, in_dim_edge, hidden_dim_edge, hidden_layers_edge, activation,
                               initializer, norm_type)
    node_model = NodeProcessor(in_dim_node, in_dim_edge, hidden_dim_node, hidden_layers_node, activation,
                               initializer, norm_type)
    return MetaLayer(edge_model=edge_model, node_model=node_model)


class GraphProcessor(nn.Module):
    """``n_iterations`` blocks applied in sequence (reference models/GNN.py:168-216)."""

    def __init__(self, n_iterations: int, in_dim_node: int, in_dim_edge: int, hidden_dim_node: int = 128,
                 hidden_dim_edge: int = 128, hidden_layers_node: int = 2, hidden_layers_edge: int = 2,
                 activation: str = "ReLU", initializer: None | str = None, norm_type="LayerNorm"):
        super().__init__()
        self.blocks = nn.ModuleList(
            build_GN_block(in_dim_node, in_dim_edge, hidden_dim_node, hidden_dim_edge, hidden_layers_node,
                           hidden_layers_edge, activation, initializer, norm_type)
            for _ in range(n_iterations))

    def forward(self, x, edge_index, edge_attr):
        for block in self.blocks:
            x, edge_attr, _ = block(x, edge_index, edge_attr)
        return x, edge_attr


_GRAPHNET_DEFAULTS = dict(
    num_global_features=0, num_local_features=3, space_dim=2, out_channels=1, n_blocks=10,
    out_dim_node=128, out_dim_edge=128,
    hidden_dim_node=128, hidden_dim_edge=128, hidden_dim_decoder=128,
    hidden_dim_processor_node=128, hidden_dim_processor_edge=128,
    hidden_layers_node=2, hidden_layers_edge=2, hidden_layers_decoder=2,
    hidden_layers_processor_node=2, hidden_layers_processor_edge=2,
    norm_type="LayerNorm", activation="ReLU", initializer=None,
)


class GraphNet(nn.Module):
    """Encode-process-decode GraphNet (reference models/GNN.py:222-309; kwargs and
    defaults :230-254)."""

    def __init__(self, **kwargs):
        super().__init__()
        c = dict(_GRAPHNET_DEFAULTS)
        c.update({k: v for k, v in kwargs.items() if k in c})
        in_dim_node = c["num_local_features"] + c["num_global_features"]
        in_dim_edge = 1 + c["space_dim"]
        self.name = "GraphNet"
        self.out_dim = c["out_channels"]
        common = dict(activation=c["activation"], initializer=c["initializer"], norm_type=c["norm_type"])
        self.node_encoder = MLP(in_dim_node, c["out_dim_node"], c["hidden_dim_node"], c["hidden_layers_node"], **common)
        self.edge_encoder = MLP(in_dim_edge, c["out_dim_edge"], c["hidden_dim_edge"], c["hidden_layers_edge"], **common)
        self.graph_processor = GraphProcessor(
            c["n_blocks"], c["out_dim_node"], c["out_dim_edge"],
            c["hidden_dim_processor_node"], c["hidden_dim_processor_edge"],
            c["hidden_layers_processor_node"], c["hidden_layers_processor_edge"], **common)
        # the decoder keeps the MLP defaults for activation and has no norm (reference :289-295)
        self.node_decoder = MLP(c["out_dim_node"], self.out_dim, c["hidden_dim_decoder"],
                                c["hidden_layers_decoder"], norm_type=None)

    # -- tensor-core inference path ------------------------------------------------
    def _tc_eligible(self) -> bool:
        """tcgen05 engine: every MLP is Linear(.,128)-ReLU-Linear(128,128)-ReLU-Linear(128,128|1)
        with LayerNorm (none on the decoder), i.e. the configuration main.py builds."""
        if ops.ENGINE != "tc":
            return False
        # recomputed on every forward (a few isinstance / shape checks): a module edited after construction - swapped
        # norm or activation, resized or re-typed layers, a half()/double() cast - must not keep dispatching here

        def mlp_ok(mlp, in_dim, out_dim, norm):
            m = list(mlp.model)
            if len(m) != (6 if norm else 5) or not all(isinstance(m[i], nn.Linear) for i in (0, 2, 4)):
                return False
            if not all(isinstance(m[i], nn.ReLU) for i in (1, 3)):
                return False
            if [tuple(m[i].weight.shape) for i in (0, 2, 4)] != [(128, in_dim), (128, 128), (out_dim, 128)]:
                return False
            if any(m[i].bias is None or m[i].weight.dtype != torch.float32 for i in (0, 2, 4)):
                return False
            if norm:
                ln = m[5]
                return isinstance(ln, nn.LayerNorm) and ln.elementwise_affine and ln.bias is not None
            return True

        ok = self.out_dim == 1 and mlp_ok(self.node_decoder, 128, 1, False)
        ok = ok and mlp_ok(self.node_encoder, self.node_encoder.model[0].in_features, 128, True)
        ok = ok and mlp_ok(self.edge_encoder, self.edge_encoder.model[0].in_features, 128, True)
        for blk in self.graph_processor.blocks:
            ok = ok and isinstance(blk.edge_model, EdgeProcessor) and isinstance(blk.node_model, NodeProcessor)
            ok = ok and mlp_ok(blk.edge_model.edge_processor, 384, 128, True)
            ok = ok and mlp_ok(blk.node_model.node_processor, 256, 128, True)
        return bool(ok)

    def _forward_tc(self, x, pos, graph: GraphIndex):
        """Same function as ``forward`` on the 3xTF32 tensor-core engine.  The first Linear of
        the edge processor is evaluated as ``e @ Wc.T + (h @ Wa.T)[row] + (h @ Wb.T)[col] + b``
        - algebraically ``cat([h[row], h[col], e]) @ W0.T + b`` with the two node-side products
        done once per node instead of once per edge - and the node processor's as
        ``agg @ Vb.T + h @ Va.T + c``; every contraction is then a [rows,128] x [128,128] tile."""
        tcl = ops.tc_linear

        def chain(a, first, mlp, n_tail=2, **kw):
            """One launch for [first +] the last ``n_tail`` Linear layers of ``mlp`` and its LayerNorm:
            the hidden activations stay on chip (csrc/tc_chain.cu)."""
            m = mlp.model
            layers = ([first] if first is not None else []) + [(m[i].weight, m[i].bias) for i in (2, 4)[2 - n_tail:]]
            if len(m) > 5:
                kw.update(gamma=m[5].weight, beta=m[5].bias, eps=m[5].eps)
            return ops.tc_mlp_chain(a, layers, **kw)

        ne, ee = self.node_encoder.model, self.edge_encoder.model
        if ne[0].in_features <= 8:       # Linear(3, 128) + ReLU folded into the launch's loader
            h = chain(x, None, self.node_encoder, narrow=(ne[0].weight, ne[0].bias))
        else:
            h = chain(ops.linear([x], ne[0].weight, ne[0].bias, relu=True), None, self.node_encoder)
        # Grid graphs from our builders: edges fall into <= 4 classes with identical geometry rows
        # (SURVEY.md 0.4), so the edge encoder runs on one row per class and the encoded edge
        # latent of block 0 is a 4-row table indexed by class - never an [E, 128] tensor.  Only
        # taken when `pos` is the very tensor the builder emitted with that topology.
        e_tab = None
        if graph.classes_valid_for(pos) and graph.class_geom.shape[1] == ee[0].in_features:
            e_tab = chain(ops.linear([graph.class_geom], ee[0].weight, ee[0].bias, relu=True), None, self.edge_encoder)
            e = None
        else:
            e = chain(ops.linear([ops.edge_geometry(pos, graph)], ee[0].weight, ee[0].bias, relu=True), None,
                      self.edge_encoder)
        # Grid graphs without diagonals (table form only): edge latents live in paired destination slots - slot 2v holds
        # node v's horizontal in-edge, 2v + 1 its vertical one, a padding slot the row +0.0 - so scatter_sum(e, col) is
        # (0 + e[2v]) + e[2v + 1] (the reference's order, bit for bit): two adjacent rows, no index.  The last block's edge
        # launch writes these node sums instead of edge latents that nothing else reads.  A form of the aggregation folded
        # into the node launch: GNC_FUSE_AGG=0 turns it off too.
        slots = graph.pair_slots if (ops.PAIRED_EDGES and ops.FUSE_AGG and e is None) else None
        blocks = self.graph_processor.blocks
        for bi, blk in enumerate(blocks):
            em = blk.edge_model.edge_processor
            nm = blk.node_model.node_processor
            W0, b0 = em.model[0].weight, em.model[0].bias
            V0, c0 = nm.model[0].weight, nm.model[0].bias
            # the two node-side products of the edge processor read the same h: one launch
            P, Q = ops.tc_linear_multi(h, [W0[:, 0:128], W0[:, 128:256]])
            if slots is not None:
                s_src, s_dst, s_cls = slots
                kw = dict(gather0=(P, s_src), gather1=(Q, s_dst), edge_slots=2 if bi == len(blocks) - 1 else 1)
                if e is None:
                    e = chain(None, None, em, pre=(tcl(e_tab, W0[:, 256:384]), s_cls, b0), residual=(e_tab, s_cls), **kw)
                else:
                    e = chain(e, (W0[:, 256:384], b0), em, residual=e, **kw)
                del P, Q
                if kw["edge_slots"] == 2:       # e holds the node sums: the plain two-operand form
                    h = chain(e, (V0[:, 128:256], c0), nm, operand2=(h, V0[:, 0:128]), residual=h)
                else:                           # the loader forms (0 + e[2m]) + e[2m + 1]
                    h = chain(e, (V0[:, 128:256], c0), nm, operand2=(h, V0[:, 0:128]), residual=h, paired=True)
                continue
            if e is None:       # block 0 in table form: e @ Wc.T is a 4-row table too
                # relu(R[class] + P[row] + Q[col] + b0) is built inside the launch as its first operand
                R = tcl(e_tab, W0[:, 256:384])
                e = chain(None, None, em, pre=(R, graph.edge_class, b0), gather0=(P, graph.src), gather1=(Q, graph.dst),
                          residual=(e_tab, graph.edge_class))
            else:               # the whole edge MLP in one launch: e Wc^T + P[row] + Q[col] + b0 -> ... -> LN + e
                e = chain(e, (W0[:, 256:384], b0), em, gather0=(P, graph.src), gather1=(Q, graph.dst), residual=e)
            del P, Q
            # the whole node MLP in one launch: cat([h, agg]) V0^T + c0 as a two-operand contraction -> ... -> LN + h
            if ops.FUSE_AGG and graph.num_edges > 0 and graph.max_in_degree() <= 2:
                # ... and scatter_sum(e, col) inside it: the loader forms agg[m] = e[eid0] + e[eid1] (same bits)
                h = chain(e, (V0[:, 128:256], c0), nm, operand2=(h, V0[:, 0:128]), residual=h,
                          agg=(graph.dst_rowptr, graph.dst_eid))
            else:
                agg = ops.aggregate(e, graph)
                h = chain(agg, (V0[:, 128:256], c0), nm, operand2=(h, V0[:, 0:128]), residual=h)
                del agg
        dec = self.node_decoder.model
        return ops.tc_mlp_chain(h, [(dec[0].weight, dec[0].bias), (dec[2].weight, dec[2].bias)],
                                dot_w=dec[4].weight, dot_b=dec[4].bias)

    def _forward_tc_train(self, x, pos, graph: GraphIndex):
        """Differentiable form of ``_forward_tc``.  The K = 3 first layers of the encoders are autograd operators of
        their own (thin streaming kernels that mask their own ReLU); everything behind them, down to the decoder's
        ``Linear(128, 1)`` row dot product, is one ``autograd.Function`` with a hand-scheduled backward
        (``tc_train.GraphNetCoreFn``: gradient sums folded into GEMM epilogues, no elementwise passes)."""
        if ops.TRAIN_PATH != "core":
            return self._forward_tc_train_opwise(x, pos, graph)
        ne, ee, dec = self.node_encoder.model, self.edge_encoder.model, self.node_decoder.model
        a1n = ops.linear([x], ne[0].weight, ne[0].bias, relu=True)
        if graph.classes_valid_for(pos) and graph.class_geom.shape[1] == ee[0].in_features:
            # Grid graphs from our builders (same condition as the inference shortcut): the edges fall into <= 4
            # classes with identical geometry rows, so the edge ENCODER - forward and backward - runs on one row per
            # class; its output is expanded to the edges by a gather and its gradient comes back as per-class sums.
            a1t = ops.linear([graph.class_geom], ee[0].weight, ee[0].bias, relu=True)
            e_tab = tc_train.MlpTailFn.apply(ee[5].eps, a1t, ee[2].weight, ee[2].bias, ee[4].weight, ee[4].bias,
                                             ee[5].weight, ee[5].bias)
            if graph.class_sum_plan is None:
                graph.class_sum_plan = tc_train.class_sum_plan(graph.edge_class, e_tab.shape[0])
            e0 = tc_train.ExpandClassRowsFn.apply(e_tab, graph.edge_class, graph.class_sum_plan)
            return tc_train.graphnet_core(self, graph, a1n, e0, edge_ready=True)
        a1e = ops.linear([ops.edge_geometry(pos, graph)], ee[0].weight, ee[0].bias, relu=True)
        return tc_train.graphnet_core(self, graph, a1n, a1e)

    def _forward_tc_train_opwise(self, x, pos, graph: GraphIndex):
        """Op-by-op autograd form (every layer its own ``autograd.Function``): the implementation the
        hand-scheduled core is tested against.  The same restructured contractions through
        ``ops.tc_linear_autograd`` (tensor-core forward and data gradients), LayerNorm and the
        K=3 / N=1 end layers through the fp32 operators, which save what their backward needs."""
        tcl = ops.tc_linear_autograd

        # ReLU backward rides in the data-gradient epilogue of the next layer (mask_input) and the
        # producing layer skips its own mask pass (premasked): every activation here has one consumer.
        def tail(a1, mlp, residual=None, a1_is_tc=True):
            m = mlp.model
            a2 = tcl(a1, m[2].weight, m[2].bias, relu=True, mask_input=a1_is_tc, premasked=True)
            z3 = tcl(a2, m[4].weight, m[4].bias, mask_input=True)
            return ops.layer_norm(z3, m[5].weight, m[5].bias, m[5].eps, residual)

        ne, ee = self.node_encoder.model, self.edge_encoder.model
        # the K = 3 first layers run on the fp32 operator, which masks its own ReLU (a1_is_tc=False)
        h = tail(ops.linear([x], ne[0].weight, ne[0].bias, relu=True), self.node_encoder, a1_is_tc=False)
        e = tail(ops.linear([ops.edge_geometry(pos, graph)], ee[0].weight, ee[0].bias, relu=True), self.edge_encoder,
                 a1_is_tc=False)
        for blk in self.graph_processor.blocks:
            em = blk.edge_model.edge_processor
            W0, b0 = em.model[0].weight, em.model[0].bias
            P = tcl(h, W0[:, 0:128])
            Q = tcl(h, W0[:, 128:256])
            a1 = tcl(e, W0[:, 256:384], b0, relu=True, P=P, Q=Q, graph=graph, premasked=True)
            e = tail(a1, em, residual=e)
            nm = blk.node_model.node_processor
            V0, c0 = nm.model[0].weight, nm.model[0].bias
            agg = ops.aggregate(e, graph)
            T = tcl(h, V0[:, 0:128])
            n1 = tcl(agg, V0[:, 128:256], c0, relu=True, addend=T, premasked=True)
            h = tail(n1, nm, residual=h)
        dec = self.node_decoder.model
        d1 = tcl(h, dec[0].weight, dec[0].bias, relu=True, premasked=True)
        d2 = tcl(d1, dec[2].weight, dec[2].bias, relu=True, mask_input=True)     # masked by its own pass
        return ops.linear([d2], dec[4].weight, dec[4].bias, relu=False)

    def forward(self, x, pos, edge_index):
        graph = edge_index if isinstance(edge_index, GraphIndex) else ops.graph_of(edge_index, x.size(0))
        if x.is_cuda and self._tc_eligible():
            if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
                return self._forward_tc_train(x, pos, graph)
            y = self._forward_tc(x, pos, graph)
            if ops.CHAIN_GUARD and not torch.cuda.is_current_stream_capturing() and not bool(torch.isfinite(y).all()):
                # an activation left the fp16 two-piece domain of the chained kernels (|a| >= 4094): same function on
                # the 3xTF32 per-layer engine, which has fp32's exponent range
                ops.CHAIN_GUARD_EVENTS += 1
                with torch.no_grad():
                    y = self._forward_tc_train_opwise(x, pos, graph)
            return y
        edge_attr = ops.edge_geometry(pos, graph)          # [pos[col]-pos[row], L1]  (reference :299-302)
        out = self.node_encoder(x)
        edge_attr = self.edge_encoder(edge_attr)
        out, _ = self.graph_processor(out, graph, edge_attr)
        return self.node_decoder(out)


class LinearClassifier(nn.Module):
    """fc1 -> ReLU -> fc2 -> ReLU -> fc3 (reference models/GNN.py:312-325)."""

    def __init__(self, in_features=128 * 128, classes=2):
        super().__init__()
        self.fc1 = nn.Linear(in_features=in_features, out_features=128)
        self.fc2 = nn.Linear(in_features=128, out_features=32)
        self.fc3 = nn.Linear(in_features=32, out_features=classes)
        self.relu = nn.ReLU()

    def forward(self, x):
        one = x.dim() == 1
        v = x.reshape(1, -1) if one else x
        v = ops.linear([v], self.fc1.weight, self.fc1.bias, relu=True)
        v = ops.linear([v], self.fc2.weight, self.fc2.bias, relu=True)
        v = ops.linear([v], self.fc3.weight, self.fc3.bias, relu=False)
        return v.reshape(-1) if one else v


class CombinedModel(nn.Module):
    """GraphNet + flatten readout + classifier head (reference models/GNN.py:327-341)."""

    def __init__(self, graph_net: Optional[GraphNet] = None, num_nodes: int = 128 * 128, classes: int = 2):
        super().__init__()
        self.graph_net = graph_net if graph_net is not None else GraphNet()
        self.num_nodes = num_nodes
        in_features = num_nodes * self.graph_net.out_dim
        self.classifier = LinearClassifier(in_features=in_features, classes=classes)

    def forward(self, x, pos=None, edge_index=None):
        if pos is None and edge_index is None and isinstance(x, tuple):
            x, pos, edge_index = x
        y = self.graph_net(x, pos, edge_index)
        topo = edge_index if isinstance(edge_index, GraphIndex) else getattr(edge_index, "_gnc_graph", None)
        if topo is not None and topo.node_ptr is not None:
            # graphs with different node counts (superpixel graphs, SURVEY.md Q7): pad / truncate each graph's node
            # outputs to num_nodes - the reference's flatten when the count matches, defined where it would crash
            if self.graph_net.out_dim != 1:
                raise NotImplementedError("the variable-size readout is defined for out_channels = 1")
            dense = ops.segment_readout(y, topo.node_ptr, self.num_nodes)
            out = self.classifier(dense)
            return out.reshape(-1) if dense.shape[0] == 1 else out
        n_graphs = y.shape[0] // self.num_nodes if y.shape[0] > self.num_nodes else 1
        if n_graphs <= 1:
            return self.classifier(y.flatten())            # [classes], as the reference
        return self.classifier(y.reshape(n_graphs, -1))    # [B, classes]
