"""Loss / optimizer kernels of the training step (csrc/train_ops.cu) and the in-place gradient accumulation of the
pipeline, against torch's own CrossEntropyLoss / Adam (what the reference's train() uses, utils/train_model.py:9-10)."""
import numpy as np
import pytest
import torch

from oracle import gnn as ognn
from oracle.weights import fill_deterministic, synthetic_images

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("B,C", [(1, 2), (7, 2), (171, 2), (300, 5)])
def test_cross_entropy_forward_backward(B, C):
    from graphnet_classifier_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(B * 10 + C)
    logits = (torch.randn(B, C, generator=g, device="cuda") * 4).requires_grad_()
    labels = torch.randint(0, C, (B,), generator=g, device="cuda")
    total = torch.full((1,), 2.5, device="cuda")
    loss = ops.cross_entropy(logits, labels, scale=1.0 / B, total=total)
    loss.backward()
    ref_in = logits.detach().double().requires_grad_()
    ref = torch.nn.functional.cross_entropy(ref_in, labels, reduction="mean")
    ref.backward()
    assert abs(loss.item() - ref.item()) < 1e-6 * max(1.0, abs(ref.item()))
    assert abs(total.item() - 2.5 - ref.item()) < 2e-6 * max(1.0, abs(ref.item()))
    assert float((logits.grad.double() - ref_in.grad).abs().max()) < 1e-7
    one = ops.cross_entropy(logits.detach()[0], labels[:1])          # [C] logits of one graph, as the reference loop has
    assert abs(one.item() - torch.nn.functional.cross_entropy(logits.detach()[0].double(), labels[0]).item()) < 1e-6


def test_adam_step_matches_torch_adam():
    from graphnet_classifier_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(0)
    n = 100003
    p0 = torch.randn(n, generator=g, device="cuda")
    ref = torch.nn.Parameter(p0.clone())
    opt = torch.optim.Adam([ref], lr=1e-3)
    p, m, v = p0.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    for step in range(1, 6):
        grad = torch.randn(n, generator=g, device="cuda") * (10.0 ** (-step))
        ref.grad = grad.clone()
        opt.step()
        ops.adam_step(p, grad * 4.0, m, v, step, lr=1e-3, grad_scale=0.25)
        assert float((p - ref.detach()).abs().max()) < 1e-6, step          # 1-2 ulp of weights of magnitude ~3
        assert torch.equal(p, ref.detach()), step                           # torch's roundings, bit for bit
    st = opt.state[ref]
    rel = lambda a, b: float((a.double() - b.double()).norm() / b.double().norm())
    assert rel(m, st["exp_avg"]) < 1e-6 and rel(v, st["exp_avg_sq"]) < 1e-6


def _model(r):
    from graphnet_classifier_b200.models.GNN import CombinedModel, GraphNet
    cfg = dict(num_local_features=3, space_dim=2, out_channels=1, n_blocks=3)
    om = ognn.OracleCombinedModel(ognn.OracleGraphNet(**cfg), num_nodes=r * r, classes=2)
    fill_deterministic(om, seed=3)
    gm = CombinedModel(GraphNet(**cfg), num_nodes=r * r, classes=2)
    gm.load_state_dict(om.state_dict())
    return gm.cuda()


def test_pipeline_step_flat_adam_equals_torch_adam_and_accumulates_in_place():
    """Three training steps of the batched pipeline with micro-batches: FlatAdam (flat parameters, one-launch update,
    gradients accumulated in place by the producing kernels, own cross-entropy kernel) against torch.optim.Adam on the
    same model with autograd's accumulation - same losses, same parameters."""
    from graphnet_classifier_b200 import ops
    from graphnet_classifier_b200.pipeline import GraphClassifierPipeline
    from graphnet_classifier_b200.utils.distributed import FlatAdam
    r, B = 16, 7
    imgs = torch.from_numpy(synthetic_images(B, r, seed=9))
    labels = torch.tensor([i % 2 for i in range(B)])
    ma, mb = _model(r), _model(r)
    pa = GraphClassifierPipeline(ma, resize_value=r, train_micro_batch=3)
    pb = GraphClassifierPipeline(mb, resize_value=r, train_micro_batch=3)
    oa = FlatAdam(ma.parameters(), lr=1e-3)
    ob = torch.optim.Adam(mb.parameters(), lr=1e-3)
    assert all(p.data_ptr() % 16 == 0 and p.grad.data_ptr() % 16 == 0 for p in ma.parameters())
    for step in range(3):
        la = pa.train_step(imgs, labels, oa)
        prev, ops.ACCUMULATE_GRADS = ops.ACCUMULATE_GRADS, False
        try:
            lb = pb.train_step(imgs, labels, ob)                 # .grad is None at step 0, autograd accumulates
        finally:
            ops.ACCUMULATE_GRADS = prev
        assert abs(la.item() - lb.item()) < 2e-6 * max(1.0, abs(lb.item())), (step, la.item(), lb.item())
        for (n, a), (_, b) in zip(ma.named_parameters(), mb.named_parameters()):
            # Adam's first steps move every weight by ~lr regardless of the gradient's size: compare absolutely
            assert float((a - b).abs().max()) < 5e-6, (step, n, float((a - b).abs().max()))
    # the in-place path was really taken: gradients live in the flat buffer and state_dict still has the reference's keys
    assert all(p.grad.data_ptr() == oa.flat[o:o + 1].data_ptr() for p, o in zip(oa.params, oa.offsets))
    assert list(ma.state_dict().keys()) == list(mb.state_dict().keys())
