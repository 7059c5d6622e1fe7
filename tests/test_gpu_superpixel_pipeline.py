"""Superpixel graphs in GraphClassifierPipeline: the fixed-capacity batch of the captured path against the exact
builder (bit for bit), its capacity bound on device SLIC outputs, and infer / infer_graphed / forward_backward /
infer_files with method="superpixel" against the hand-assembled path and the per-graph oracle."""
import numpy as np
import pytest
import torch
from PIL import Image

from oracle import gnn as ognn
from oracle import graph_build as ogb
from oracle.weights import fill_deterministic

pytestmark = pytest.mark.gpu

CFG = dict(num_local_features=3, space_dim=2, out_channels=1, n_blocks=3)


def _smooth_images(rng, B, H, W, noise=6):
    low = rng.random((B, 5, 5, 3))
    img = np.kron(low, np.ones((1, H // 5 + 1, W // 5 + 1, 1)))[:, :H, :W]
    return np.clip(img * 255 + rng.integers(-noise, noise + 1, (B, H, W, 3)), 0, 255).astype(np.uint8)


def _voronoi(rng, H, W, k):
    seeds = rng.random((k, 2)) * [H, W]
    yy, xx = np.mgrid[0:H, 0:W]
    return ((yy[..., None] - seeds[:, 0]) ** 2 + (xx[..., None] - seeds[:, 1]) ** 2).argmin(-1).astype(np.int32)


def _bits(t):
    return t.contiguous().view(torch.int32) if t.dtype == torch.float32 else t


def _check_padded_equals_exact(img, lab, S_cap, E_cap):
    from graphnet_classifier_b200.utils.image_to_graph.batched import build_superpixel_batch, build_superpixel_batch_padded
    B = img.shape[0]
    ex = build_superpixel_batch(img, labels=lab)
    pad, flag = build_superpixel_batch_padded(img, lab, S_cap, E_cap)
    assert int(flag.item()) == 0
    n, e = ex.x.shape[0], ex.edge_index.shape[1]
    N, E = B * S_cap + 1, B * E_cap
    assert pad.x.shape == (N, 3) and pad.pos.shape == (N, 2) and pad.edge_index.shape == (2, E)
    g, gx = pad.graph, ex.graph
    assert torch.equal(g.node_ptr, gx.node_ptr) and int(g.node_ptr[-1]) == n
    # real rows and edges: the exact batch's, bit for bit
    assert torch.equal(_bits(pad.x[:n]), _bits(ex.x)) and torch.equal(_bits(pad.pos[:n]), _bits(ex.pos))
    assert torch.equal(pad.edge_index[:, :e], ex.edge_index)
    # padding: zero rows, self-loops on the padding rows, spread round robin
    assert not _bits(pad.x[n:]).any() and not _bits(pad.pos[n:]).any()
    k = torch.arange(E - e, device=img.device)
    loops = n + k % (N - n)
    assert torch.equal(pad.edge_index[0, e:], loops) and torch.equal(pad.edge_index[1, e:], loops)
    # CSR of the real nodes: the same in-edges (and out-edges) in the same order
    for rp, eid, rpx, eidx in ((g.dst_rowptr, g.dst_eid, gx.dst_rowptr, gx.dst_eid),
                               (g.src_rowptr, g.src_eid, gx.src_rowptr, gx.src_eid)):
        assert torch.equal(rp[:n + 1], rpx) and torch.equal(eid[:e], eidx)
    return ex, pad


def test_padded_batch_equals_exact_on_slic_and_supplied_labels(libgnc):
    from graphnet_classifier_b200.utils.image_to_graph.batched import build_superpixel_graphs, superpixel_capacity
    from graphnet_classifier_b200.utils.image_to_graph.slic import connectivity_min_size, slic_labels
    rng = np.random.default_rng(11)
    # SLIC labels at the pipeline's capacities
    for (B, r, ns) in ((3, 64, 30), (2, 40, 100), (1, 8, 100)):
        img = torch.from_numpy(_smooth_images(rng, B, r, r)).cuda()
        lab = slic_labels(img, n_segments=ns)
        _check_padded_equals_exact(img, lab, *superpixel_capacity(r, r, connectivity_min_size(r, r, ns)))
    # supplied maps: Voronoi cells, one of them with two labels merged into one disconnected label, caps just fitting
    B, H, W = 4, 36, 52
    img = torch.from_numpy(_smooth_images(rng, B, H, W)).cuda()
    labs = [_voronoi(rng, H, W, k) for k in (9, 23, 31, 14)]
    far = labs[1][0, 0], labs[1][-1, -1]
    assert far[0] != far[1]
    labs[1] = np.where(labs[1] == far[1], far[0], labs[1])
    labs = [np.unique(lb, return_inverse=True)[1].reshape(H, W).astype(np.int32) for lb in labs]     # labels 0 .. S - 1
    lab = torch.from_numpy(np.stack(labs)).cuda()
    n_nodes, _, _, n_edges, _ = build_superpixel_graphs(img, lab)
    S, E = int(n_nodes.max()), int(n_edges.max())
    _check_padded_equals_exact(img, lab, S, E)
    _check_padded_equals_exact(img, lab, S + 7, E + 30)


def test_padded_batch_flags_exactly_the_exceeded_cap(libgnc):
    from graphnet_classifier_b200.utils.image_to_graph.batched import build_superpixel_batch_padded, build_superpixel_graphs
    rng = np.random.default_rng(2)
    B, H, W = 3, 32, 40
    img = torch.from_numpy(_smooth_images(rng, B, H, W)).cuda()
    lab = torch.from_numpy(np.stack([_voronoi(rng, H, W, k) for k in (12, 20, 7)])).cuda()
    n_nodes, _, _, n_edges, _ = build_superpixel_graphs(img, lab)
    S, E = int(n_nodes.max()), int(n_edges.max())

    def flag(lb, s, e):
        return int(build_superpixel_batch_padded(img, lb, s, e)[1].item())
    assert flag(lab, S, E) == 0
    assert flag(lab, S - 1, E) == 1                  # label S - 1 above max_label = S_cap - 1
    assert flag(lab, S, E - 1) == 4
    bad = lab.clone()
    bad[2, 5, 7] = 1 << 30
    assert flag(bad, S, E) == 1
    bad[0, 0, 0] = -3
    assert flag(bad, S, E) == 1


def test_padded_entry_point_never_writes_outside_its_buffers(libgnc):
    """The C entry point on hostile inputs (offsets past the buffers, negative, counts over the caps, wild labels):
    every element around the output buffers keeps its sentinel, and the flag reports the overflow."""
    from graphnet_classifier_b200.ops import _stream
    B, S_cap, E_cap, H, W = 3, 5, 8, 4, 4
    dev = "cuda"
    x = torch.rand(B, S_cap, 3, device=dev)
    pos = torch.rand(B, S_cap, 2, device=dev)
    edges = torch.randint(0, S_cap, (B, 2, E_cap), dtype=torch.int64, device=dev)
    n_nodes = torch.tensor([9, 2, 5], dtype=torch.int32, device=dev)
    n_edges = torch.tensor([3, 100, 8], dtype=torch.int32, device=dev)
    labels = torch.tensor([-1, 7, 1 << 30, 2] * (B * H), dtype=torch.int32, device=dev)
    node_ptr = torch.tensor([-5, 40, 3, 1 << 30], dtype=torch.int32, device=dev)
    edge_ptr = torch.tensor([2, -7, 1 << 40, 30], dtype=torch.int64, device=dev)
    N, E, G = B * S_cap + 1, B * E_cap, 64
    xb = torch.full((N * 3 + 2 * G,), float("nan"), device=dev)
    pb = torch.full((N * 2 + 2 * G,), float("nan"), device=dev)
    eb = torch.full((2 * E + 2 * G,), -99, dtype=torch.int64, device=dev)
    ov = torch.full((3,), -99, dtype=torch.int32, device=dev)
    rc = libgnc.gnc_superpixel_batch_padded(x.data_ptr(), pos.data_ptr(), edges.data_ptr(), n_nodes.data_ptr(),
                                            n_edges.data_ptr(), labels.data_ptr(), B, H, W, S_cap - 1, S_cap, E_cap,
                                            node_ptr.data_ptr(), edge_ptr.data_ptr(), xb[G:].data_ptr(), pb[G:].data_ptr(),
                                            eb[G:].data_ptr(), ov[1:].data_ptr(), _stream())
    assert rc == 0
    torch.cuda.synchronize()
    for buf, n in ((xb, N * 3), (pb, N * 2)):
        assert torch.isnan(buf[:G]).all() and torch.isnan(buf[G + n:]).all()
    assert (eb[:G] == -99).all() and (eb[G + 2 * E:] == -99).all()
    assert int(ov[0]) == -99 and int(ov[2]) == -99 and int(ov[1]) == 1 | 2 | 4


@pytest.mark.parametrize("B,H,W,ns", [(4, 256, 256, 100), (6, 128, 128, 100), (4, 64, 48, 30), (3, 33, 50, 20),
                                      (4, 16, 16, 100), (4, 8, 8, 100), (3, 5, 7, 50)])
def test_slic_graphs_stay_within_capacity(libgnc, B, H, W, ns):
    """The bound the captured path relies on, on device SLIC outputs: smooth images and pure noise (the most regions),
    down to images so small that min_size is 0."""
    from graphnet_classifier_b200.utils.image_to_graph.batched import build_superpixel_graphs, superpixel_capacity
    from graphnet_classifier_b200.utils.image_to_graph.slic import connectivity_min_size, slic_labels
    rng = np.random.default_rng(H * W + ns)
    m = connectivity_min_size(H, W, ns)
    S_cap, E_cap = superpixel_capacity(H, W, m)
    for img in (_smooth_images(rng, B, H, W), rng.integers(0, 256, (B, H, W, 3), dtype=np.uint8)):
        lab = slic_labels(torch.from_numpy(img).cuda(), n_segments=ns)
        n_nodes, _, _, n_edges, _ = build_superpixel_graphs(torch.from_numpy(img), lab)
        assert int(lab.min()) >= 0 and int(lab.max()) <= S_cap - 1
        assert int(n_nodes.max()) <= S_cap and int(n_edges.max()) <= E_cap, (m, S_cap, E_cap, n_nodes, n_edges)


def _models(num_nodes, seed=17):
    from graphnet_classifier_b200.models.GNN import CombinedModel, GraphNet
    om = ognn.OracleCombinedModel(ognn.OracleGraphNet(**CFG), num_nodes=num_nodes, classes=2)
    fill_deterministic(om, seed=seed)
    gm = CombinedModel(GraphNet(**CFG), num_nodes=num_nodes, classes=2)
    gm.load_state_dict(om.state_dict())
    return om, gm.cuda()


def test_infer_equals_hand_assembled_path_and_oracle(libgnc):
    from graphnet_classifier_b200.pipeline import GraphClassifierPipeline
    from graphnet_classifier_b200.utils.image_to_graph.batched import build_superpixel_batch
    from graphnet_classifier_b200.utils.image_to_graph.slic import slic_labels
    r, B, ns = 48, 5, 30
    om, gm = _models(num_nodes=30)
    rng = np.random.default_rng(7)
    imgs = np.concatenate([_smooth_images(rng, 1, r, r, noise=n) for n in (2, 20, 45, 70, 100)])
    pipe = GraphClassifierPipeline(gm, r, method="superpixel", n_segments=ns)
    got = pipe.infer(torch.from_numpy(imgs))
    img = torch.from_numpy(imgs).cuda()
    lab = slic_labels(img, n_segments=ns)
    with torch.no_grad():
        exp = gm(build_superpixel_batch(img, labels=lab).as_tuple())
    assert got.shape == (B, 2) and torch.equal(got, exp)
    ln = lab.cpu().numpy()
    graphs = [ogb.to_model_inputs(*ogb.superpixel_graph_from_labels(imgs[b], ln[b].astype(np.int64))) for b in range(B)]
    counts = [g[0].shape[0] for g in graphs]
    assert len(set(counts)) > 1, counts
    with torch.no_grad():
        ref = ognn.padded_readout_logits(om, graphs)
    np.testing.assert_allclose(got.cpu().numpy(), ref.numpy(), rtol=1e-5, atol=1e-6)
    # micro-batches (2 + 2 + 1) give the same logits
    pipe_mb = GraphClassifierPipeline(gm, r, method="superpixel", n_segments=ns, micro_batch=2)
    assert torch.equal(pipe_mb.infer(torch.from_numpy(imgs)), got)


def test_infer_graphed_equals_infer_and_overflow_falls_back(libgnc):
    from graphnet_classifier_b200 import ops
    from graphnet_classifier_b200.pipeline import GraphClassifierPipeline
    from graphnet_classifier_b200.utils.image_to_graph.batched import build_superpixel_batch
    from graphnet_classifier_b200.utils.image_to_graph.slic import slic_labels
    torch.manual_seed(3)
    r, ns = 64, 40
    _, gm = _models(num_nodes=40, seed=5)
    gm.eval()
    pipe = GraphClassifierPipeline(gm, r, method="superpixel", n_segments=ns)
    rng = np.random.default_rng(9)
    for B in (1, 3):
        sizes = set()
        for noise in (2, 40, 90):            # different images: different node and edge counts through one capture
            imgs = torch.from_numpy(_smooth_images(rng, B, r, r, noise=noise))
            got = pipe.infer_graphed(imgs)
            assert torch.equal(got, pipe.infer(imgs))
            gb = build_superpixel_batch(imgs.cuda(), labels=slic_labels(imgs.cuda(), n_segments=ns))
            sizes.add((gb.x.shape[0], gb.edge_index.shape[1]))
        assert len(sizes) == 3, sizes
    assert len(pipe._graphs) == 2
    # updated weights are read at replay time
    with torch.no_grad():
        for prm in gm.parameters():
            prm.mul_(1.01)
    imgs = torch.from_numpy(_smooth_images(rng, 3, r, r))
    assert torch.equal(pipe.infer_graphed(imgs), pipe.infer(imgs))
    # a capacity below what these images need: the flag is set and the call returns the exact builder's logits
    before = ops.SUPERPIXEL_OVERFLOW_EVENTS
    pipe.superpixel_caps = (6, 18)
    got = pipe.infer_graphed(imgs)
    assert ops.SUPERPIXEL_OVERFLOW_EVENTS == before + 1
    assert torch.equal(got, pipe.infer(imgs))


def _oracle64_grads(om, graphs, lab):
    """The oracle's gradients in float64 (its MLPs keep float64 instead of the reference's fp32 cast), for the ReLU-tie
    rule of DESIGN.md section 6: a tensor passes at max(1e-5, 3 x |oracle32 - oracle64|)."""
    import copy
    om64 = copy.deepcopy(om).double()
    for mlp in [m for m in om64.modules() if isinstance(m, ognn.OracleMLP)]:
        mlp.forward = (lambda x, mlp=mlp: mlp.model(x.reshape(x.shape[0], -1)))
    om64.zero_grad()
    g64 = [tuple(t.double() if t.is_floating_point() else t for t in g) for g in graphs]
    torch.nn.functional.cross_entropy(ognn.padded_readout_logits(om64, g64), lab).backward()
    return {n: p.grad for n, p in om64.named_parameters()}


def test_forward_backward_and_train_step_match_hand_path_and_oracle(libgnc):
    from graphnet_classifier_b200 import ops
    from graphnet_classifier_b200.pipeline import GraphClassifierPipeline
    from graphnet_classifier_b200.utils.image_to_graph.batched import build_superpixel_batch
    from graphnet_classifier_b200.utils.image_to_graph.slic import slic_labels
    r, B, ns = 40, 4, 25
    om, gm = _models(num_nodes=24, seed=23)
    rng = np.random.default_rng(13)
    imgs = np.concatenate([_smooth_images(rng, 1, r, r, noise=n) for n in (3, 30, 60, 90)])
    labels = np.array([0, 1, 1, 0])
    pipe = GraphClassifierPipeline(gm, r, method="superpixel", n_segments=ns)
    assert pipe.train_micro_batch >= B
    for p in gm.parameters():
        p.grad = None
    loss = pipe.forward_backward(torch.from_numpy(imgs), torch.from_numpy(labels))
    got = {n: p.grad.clone() for n, p in gm.named_parameters()}
    assert len(got) == 76
    # the same model on the same batch, assembled by hand
    for p in gm.parameters():
        p.grad = None
    img = torch.from_numpy(imgs).cuda()
    lab_map = slic_labels(img, n_segments=ns)
    gb = build_superpixel_batch(img, labels=lab_map)
    y = torch.from_numpy(labels).cuda()
    total = torch.zeros(1, dtype=torch.float32, device="cuda")
    ops.ACCUMULATE_GRADS = True
    try:
        ops.cross_entropy(gm(gb.as_tuple()), y, scale=1.0 / B, total=total).backward()
    finally:
        ops.ACCUMULATE_GRADS = False
    assert torch.equal(_bits(loss.reshape(1)), _bits(total))
    for n, p in gm.named_parameters():
        assert torch.equal(_bits(got[n]), _bits(p.grad)), n
    # the per-graph oracle on the device labels
    ln = lab_map.cpu().numpy()
    graphs = [ogb.to_model_inputs(*ogb.superpixel_graph_from_labels(imgs[b], ln[b].astype(np.int64))) for b in range(B)]
    om.zero_grad()
    lo = torch.nn.functional.cross_entropy(ognn.padded_readout_logits(om, graphs), torch.from_numpy(labels))
    lo.backward()
    assert abs(loss.item() - lo.item()) < 1e-5 * max(1.0, lo.item())
    g64 = _oracle64_grads(om, graphs, torch.from_numpy(labels))

    def rel(a, b):
        a, b = a.detach().double().cpu(), b.detach().double().cpu()
        return float((a - b).norm() / b.norm().clamp_min(1e-30))
    for (n, po) in om.named_parameters():
        noise = rel(po.grad, g64[n])
        err = min(rel(got[n], po.grad), rel(got[n], g64[n]))
        assert err < max(1e-5, 3 * noise), (n, err, noise)
    # train_step: the same loss and gradients (accumulated in place into zeroed storage: equal values), then the step
    opt = torch.optim.SGD(gm.parameters(), lr=0.0)
    loss2 = pipe.train_step(torch.from_numpy(imgs), torch.from_numpy(labels), opt)
    assert torch.equal(_bits(loss2.reshape(1)), _bits(total))
    for n, p in gm.named_parameters():
        assert torch.equal(got[n], p.grad), n


def test_infer_files_superpixel_equals_infer(libgnc, tmp_path):
    from graphnet_classifier_b200.pipeline import GraphClassifierPipeline
    from graphnet_classifier_b200.utils.staging import infer_files
    rng = np.random.default_rng(21)
    r = 48
    paths = []
    for i, (h, w) in enumerate([(60, 80), (48, 48), (90, 70), (33, 41), (64, 64)]):
        low = rng.integers(0, 256, (h // 10 + 2, w // 10 + 2, 3), dtype=np.uint8)
        im = Image.fromarray(low).resize((w, h), Image.BILINEAR)
        p = tmp_path / (f"s{i}.jpg" if i % 2 else f"s{i}.png")
        im.save(p, quality=90) if p.suffix == ".jpg" else im.save(p)
        paths.append(str(p))
    _, gm = _models(num_nodes=30, seed=4)
    pipe = GraphClassifierPipeline(gm, r, method="superpixel", n_segments=30)
    got = infer_files(pipe, paths, chunk=2)
    px = np.stack([np.array(Image.open(p).convert("RGB").resize((r, r))) for p in paths])
    assert torch.equal(got, pipe.infer(torch.from_numpy(px)))
