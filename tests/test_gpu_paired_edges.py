"""GPU: edge latents in paired destination slots (GraphIndex.pair_slots).  The slot-order edge launches equal the edge-order
launches row for row with padding slots exactly +0.0, the pair-sum output equals the aggregation of the edge-order output,
the paired node launch equals the index-driven one, and the model's logits do not change - all bit for bit."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

# (B, image H, image W, patch): ragged last tiles, H != W, one and several graphs, pixel and patch grids, several tiles per
# CTA pair
SHAPES = [(1, 13, 29, 0), (3, 40, 23, 0), (3, 64, 48, 8), (1, 1, 37, 0), (3, 128, 96, 0)]


def _graph(B, H, W, patch):
    from graphnet_classifier_b200.utils.image_to_graph.batched import build_patch_graphs, build_pixel_graphs
    rng = np.random.default_rng(B * 1000 + H * 10 + W)
    img = torch.from_numpy(rng.integers(0, 256, (B, H, W, 3), dtype=np.uint8))
    gb = build_patch_graphs(img, patch, use_cache=False) if patch else build_pixel_graphs(img, use_cache=False)
    return gb.graph


def _slot_eid(graph):
    """Edge id held by every slot (-1: padding), from the destination CSR: a node's in-edges in ascending id."""
    s_src = graph.pair_slots[0].long()
    rp, eid = graph.dst_rowptr.long(), graph.dst_eid.long()
    has_h, has_v = s_src[0::2] >= 0, s_src[1::2] >= 0
    out = torch.full_like(s_src, -1)
    first = rp[:-1]
    out[0::2] = torch.where(has_h, eid[first.clamp(max=max(eid.numel() - 1, 0))], -1)
    second = (first + has_h.long()).clamp(max=max(eid.numel() - 1, 0))
    out[1::2] = torch.where(has_v, eid[second], -1)
    return out


def _layers(gen, n, scale=11.0):
    return [((torch.randn(128, 128, generator=gen) / scale).cuda(), (torch.randn(128, generator=gen) * 0.3).cuda())
            for _ in range(n)]


def _is_pos_zero(t):
    return bool((t.contiguous().view(torch.int32) == 0).all())


@pytest.mark.parametrize("B,H,W,patch", SHAPES)
def test_slot_arrays_describe_the_edges(libgnc, B, H, W, patch):
    g = _graph(B, H, W, patch)
    s_src, s_dst, s_cls = (t.long() for t in g.pair_slots)
    assert s_src.numel() == 2 * g.num_nodes
    se = _slot_eid(g)
    real = se >= 0
    assert torch.equal(real, s_src >= 0)
    assert torch.equal(torch.sort(se[real]).values, torch.arange(g.num_edges, device=se.device))
    assert torch.equal(g.src.long()[se[real]], s_src[real])
    assert torch.equal(g.dst.long()[se[real]], s_dst[real])
    assert torch.equal(s_dst, torch.arange(2 * g.num_nodes, device=se.device) >> 1)
    assert torch.equal(g.edge_class.long()[se[real]], s_cls[real])


@pytest.mark.parametrize("B,H,W,patch", SHAPES)
def test_slot_order_edge_launch_and_pair_sums(libgnc, B, H, W, patch):
    """Three-layer edge form (blocks >= 1): slot rows = edge rows, padding +0.0; pair sums = ops.aggregate."""
    from graphnet_classifier_b200 import ops
    g = _graph(B, H, W, patch)
    gen = torch.Generator().manual_seed(B + H + W)
    N, E = g.num_nodes, g.num_edges
    se = _slot_eid(g)
    real = se >= 0
    e = (torch.randn(E, 128, generator=gen) * 2).cuda()
    e_slot = torch.zeros(2 * N, 128, device="cuda")
    e_slot[real] = e[se[real]]
    P, Q = torch.randn(N, 128, generator=gen).cuda(), torch.randn(N, 128, generator=gen).cuda()
    W0 = (torch.randn(128, 384, generator=gen) / 20).cuda()
    b0 = (torch.randn(128, generator=gen) * 0.3).cuda()
    layers = [(W0[:, 256:384], b0)] + _layers(gen, 2)
    gamma, beta = (torch.rand(128, generator=gen) + 0.5).cuda(), (torch.randn(128, generator=gen) * 0.2).cuda()
    kw = dict(gamma=gamma, beta=beta)
    ref = ops.tc_mlp_chain(e, layers, gather0=(P, g.src), gather1=(Q, g.dst), residual=e, **kw)
    s_src, s_dst, _ = g.pair_slots
    got = ops.tc_mlp_chain(e_slot, layers, gather0=(P, s_src), gather1=(Q, s_dst), residual=e_slot, edge_slots=1, **kw)
    assert got.shape == (2 * N, 128)
    assert torch.equal(got[real], ref[se[real]])
    assert _is_pos_zero(got[~real])
    sums = ops.tc_mlp_chain(e_slot, layers, gather0=(P, s_src), gather1=(Q, s_dst), residual=e_slot, edge_slots=2, **kw)
    assert sums.shape == (N, 128)
    assert torch.equal(sums, ops.aggregate(ref, g))


@pytest.mark.parametrize("B,H,W,patch", SHAPES)
def test_slot_order_prestage_launch_and_pair_sums(libgnc, B, H, W, patch):
    """Pre-stage form (block 0: edge latents as a per-class table)."""
    from graphnet_classifier_b200 import ops
    g = _graph(B, H, W, patch)
    gen = torch.Generator().manual_seed(7 * B + H + W)
    N = g.num_nodes
    se = _slot_eid(g)
    real = se >= 0
    R = torch.randn(4, 128, generator=gen).cuda()
    e_tab = torch.randn(4, 128, generator=gen).cuda()
    P, Q = torch.randn(N, 128, generator=gen).cuda(), torch.randn(N, 128, generator=gen).cuda()
    b0 = (torch.randn(128, generator=gen) * 0.3).cuda()
    layers = _layers(gen, 2)
    gamma, beta = (torch.rand(128, generator=gen) + 0.5).cuda(), (torch.randn(128, generator=gen) * 0.2).cuda()
    kw = dict(gamma=gamma, beta=beta)
    ref = ops.tc_mlp_chain(None, layers, pre=(R, g.edge_class, b0), gather0=(P, g.src), gather1=(Q, g.dst),
                           residual=(e_tab, g.edge_class), **kw)
    s_src, s_dst, s_cls = g.pair_slots
    slot_kw = dict(pre=(R, s_cls, b0), gather0=(P, s_src), gather1=(Q, s_dst), residual=(e_tab, s_cls), **kw)
    got = ops.tc_mlp_chain(None, layers, edge_slots=1, **slot_kw)
    assert torch.equal(got[real], ref[se[real]])
    assert _is_pos_zero(got[~real])
    sums = ops.tc_mlp_chain(None, layers, edge_slots=2, **slot_kw)
    assert torch.equal(sums, ops.aggregate(ref, g))


@pytest.mark.parametrize("B,H,W,patch", SHAPES)
def test_paired_node_launch_equals_index_driven(libgnc, B, H, W, patch):
    from graphnet_classifier_b200 import ops
    g = _graph(B, H, W, patch)
    gen = torch.Generator().manual_seed(3 * B + H * W)
    N, E = g.num_nodes, g.num_edges
    se = _slot_eid(g)
    real = se >= 0
    e = (torch.randn(E, 128, generator=gen) * 2).cuda()
    e_slot = torch.zeros(2 * N, 128, device="cuda")
    e_slot[real] = e[se[real]]
    h = torch.randn(N, 128, generator=gen).cuda()
    V0 = (torch.randn(128, 256, generator=gen) / 16).cuda()
    c0 = (torch.randn(128, generator=gen) * 0.2).cuda()
    layers = [(V0[:, 128:256], c0)] + _layers(gen, 2)
    gamma, beta = (torch.rand(128, generator=gen) + 0.5).cuda(), (torch.randn(128, generator=gen) * 0.2).cuda()
    kw = dict(operand2=(h, V0[:, 0:128]), gamma=gamma, beta=beta, residual=h)
    ref = ops.tc_mlp_chain(e, layers, agg=(g.dst_rowptr, g.dst_eid), **kw)
    got = ops.tc_mlp_chain(e_slot, layers, paired=True, **kw)
    assert got.shape == (N, 128) and torch.isfinite(got).all()
    assert torch.equal(got, ref)


@pytest.mark.parametrize("r,patch", [(24, 0), (40, 8)])
def test_model_logits_unchanged_eager_and_graphed(libgnc, monkeypatch, r, patch):
    from graphnet_classifier_b200 import ops
    from graphnet_classifier_b200.models.GNN import CombinedModel, GraphNet
    from graphnet_classifier_b200.pipeline import GraphClassifierPipeline
    torch.manual_seed(11)
    n = (r // patch) ** 2 if patch else r * r
    model = CombinedModel(GraphNet(num_local_features=3, space_dim=2, out_channels=1, n_blocks=3), num_nodes=n).cuda().eval()
    outs = {}
    for flag in (False, True):
        monkeypatch.setattr(ops, "PAIRED_EDGES", flag)
        pipe = GraphClassifierPipeline(model, resize_value=r, method="patch" if patch else "pixel", patch_size=patch or 8)
        for B in (1, 3):
            img = torch.from_numpy(np.random.default_rng(B).integers(0, 256, (B, r, r, 3), dtype=np.uint8))
            outs[(flag, B, "eager")] = pipe.infer(img)
            outs[(flag, B, "graphed")] = pipe.infer_graphed(img)
    for B in (1, 3):
        ref = outs[(False, B, "eager")]
        assert torch.isfinite(ref).all()
        for k in ((False, B, "graphed"), (True, B, "eager"), (True, B, "graphed")):
            assert torch.equal(outs[k], ref), k
