#!/usr/bin/env python
"""Superpixel graphs through GraphClassifierPipeline(method="superpixel"), timed on one GPU.

1. Config 4 (resize 256, 1024 images, n_segments 100): ``pipe.infer`` against the hand-assembled path of
   scripts/config4_bench.py (slic_labels -> build_superpixel_batch -> CombinedModel), interleaved, L2 flushed before
   every call.  CUDA events around each call.
2. Latency: ``infer_graphed`` (one CUDA graph per shape, replayed) against eager ``infer`` at B = 1 and B = 8,
   interleaved.  Host clock from a synchronised start to the call's result on the host side (both calls end in a
   synchronisation: ``infer`` reads the builder's output sizes back, ``infer_graphed`` its capacity flag; a final
   synchronize covers the remaining kernels).

Prints the GPU's name and power limit first.  Usage: superpixel_pipeline_bench.py [reps]
"""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from graphnet_classifier_b200 import ops
from graphnet_classifier_b200.models.GNN import CombinedModel, GraphNet
from graphnet_classifier_b200.pipeline import GraphClassifierPipeline
from graphnet_classifier_b200.utils.image_to_graph.batched import build_superpixel_batch
from graphnet_classifier_b200.utils.image_to_graph.slic import slic_labels

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 9
dev = "cuda"
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip().splitlines()
print(f"GPU: {q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()}  (name, power limit, max SM clock)")


def images(B, r, seed):
    # smooth random images (low-frequency blobs + noise), as scripts/config4_bench.py
    g = torch.Generator(device=dev).manual_seed(seed)
    low = torch.rand(B, 3, 8, 8, device=dev, generator=g)
    im = torch.nn.functional.interpolate(low, size=(r, r), mode="bilinear", align_corners=False)
    im = (im + 0.05 * torch.randn(B, 3, r, r, device=dev, generator=g)).clamp(0, 1)
    return im.mul(255).byte().permute(0, 2, 3, 1).contiguous()


def med(v):
    v = sorted(v)
    return v[len(v) // 2]


torch.manual_seed(0)
r = 256
net = CombinedModel(GraphNet(num_local_features=3, space_dim=2, out_channels=1, n_blocks=3), num_nodes=r // 2,
                    classes=2).cuda().eval()
pipe = GraphClassifierPipeline(net, r, method="superpixel", n_segments=100, compactness=10.0)
print(f"pipeline: superpixel capacities per image S_cap={pipe.superpixel_caps[0]} nodes, E_cap={pipe.superpixel_caps[1]} "
      f"edges; micro_batch {pipe.micro_batch}")

# -- 1. config 4 throughput ------------------------------------------------------------------------------------------
B = 1024
imgs = images(B, r, 0)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def hand():
    labels = slic_labels(imgs, n_segments=100, compactness=10.0)
    gb = build_superpixel_batch(imgs, labels=labels, max_nodes=128)
    with torch.no_grad():
        return net(gb.as_tuple())


def timed(fn):
    flush.zero_()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    out = fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e), out


arms = {"pipe.infer": lambda: pipe.infer(imgs), "hand-assembled (config4_bench)": hand}
for fn in arms.values():
    for _ in range(2):
        timed(fn)
res = {k: [] for k in arms}
outs = {}
for _ in range(REPS):
    for k, fn in arms.items():
        t, outs[k] = timed(fn)
        res[k].append(t)
gb = build_superpixel_batch(imgs, labels=slic_labels(imgs, n_segments=100))
counts = (gb.graph.node_ptr[1:] - gb.graph.node_ptr[:-1])
print(f"\nconfig 4: {B} images, resize {r}, n_segments 100: {gb.x.shape[0] / B:.1f} nodes (max {int(counts.max())}), "
      f"{gb.edge_index.shape[1] / B:.1f} edges per image; {REPS} interleaved calls per arm, L2 flushed before each")
for k, v in res.items():
    print(f"  {k:32s} median {med(v):8.3f} ms  min {min(v):8.3f}  max {max(v):8.3f}  -> {B / med(v) * 1e3:,.0f} images/s")
a, b = outs.values()
print(f"  logits equal between the arms: {torch.equal(a, b)} (the hand path truncates graphs to 128 nodes; "
      f"max nodes here {int(counts.max())})")

# -- 2. small-batch latency -------------------------------------------------------------------------------------------
print("\nlatency: infer_graphed (captured once per shape, replayed) vs eager infer; host clock, synchronised")
for Bs in (1, 8):
    sets = [images(Bs, r, 100 + i) for i in range(4)]
    same = all(torch.equal(pipe.infer_graphed(s), pipe.infer(s)) for s in sets)
    ev0 = ops.SUPERPIXEL_OVERFLOW_EVENTS
    lat = {"infer_graphed": [], "infer": []}
    fns = {"infer_graphed": pipe.infer_graphed, "infer": pipe.infer}
    for _ in range(3):
        for fn in fns.values():
            fn(sets[0])
    for i in range(10 * REPS):
        s = sets[i % len(sets)]
        for k, fn in fns.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn(s)
            torch.cuda.synchronize()
            lat[k].append((time.perf_counter() - t0) * 1e3)
    g, e = med(lat["infer_graphed"]), med(lat["infer"])
    print(f"  B={Bs}: infer_graphed median {g:7.3f} ms (min {min(lat['infer_graphed']):.3f})   infer median {e:7.3f} ms "
          f"(min {min(lat['infer']):.3f})   ratio {e / g:.2f}x   bit-equal on 4 image sets: {same}   "
          f"overflow fallbacks: {ops.SUPERPIXEL_OVERFLOW_EVENTS - ev0}")
