#!/usr/bin/env python
"""Micro-benchmark of the paired-slot launches (GraphIndex.pair_slots) against the edge-order launches they replace, on
the shapes of one GraphNet block at the headline configuration (512 pixel grids of 128 x 128; CUDA events, L2 flushed).
Cases are interleaved and repeated - the GPU runs at its power cap and what ran just before shifts the clocks - and
the median of the per-round best is reported.  Usage: paired_microbench.py [B]"""
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from graphnet_classifier_b200 import _lib, ops
from graphnet_classifier_b200.utils.image_to_graph.batched import build_pixel_graphs


def timeit(fn, n=3):
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); fn(); e.record(); torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    return min(ts)


_lib.load()
B = int(sys.argv[1]) if len(sys.argv) > 1 else 512
r = 128
img = torch.from_numpy(np.random.default_rng(0).integers(0, 256, (B, r, r, 3), dtype=np.uint8))
g = build_pixel_graphs(img, use_cache=False).graph
N, E = g.num_nodes, g.num_edges
s_src, s_dst, _ = g.pair_slots
dev = "cuda"
gen = torch.Generator(device=dev).manual_seed(0)
mk = lambda *s: torch.randn(*s, device=dev, generator=gen)
layers = [(mk(128, 128) / 11, mk(128) * 0.1) for _ in range(3)]
gamma, beta = torch.ones(128, device=dev), torch.zeros(128, device=dev)
P, Q, h = mk(N, 128), mk(N, 128), mk(N, 128)
e = mk(E, 128)
e_slot = torch.zeros(2 * N, 128, device=dev)
e_slot[s_src.long() >= 0] = mk(E, 128)
out_e, out_s, out_n = torch.empty(E, 128, device=dev), torch.empty(2 * N, 128, device=dev), torch.empty(N, 128, device=dev)
agg = ops.aggregate(e, g)
LN = dict(gamma=gamma, beta=beta)
node_kw = dict(operand2=(h, layers[0][0]), residual=h, out=out_n, **LN)
row = 4.0 * 128
cases = {   # name: (fn, bytes the launch has to move)
    "edge launch, edge order": (lambda: ops.tc_mlp_chain(e, layers, gather0=(P, g.src), gather1=(Q, g.dst), residual=e,
                                                         out=out_e, **LN), row * (3 * E + 2 * N)),
    "edge launch, slot order": (lambda: ops.tc_mlp_chain(e_slot, layers, gather0=(P, s_src), gather1=(Q, s_dst),
                                                         residual=e_slot, out=out_s, edge_slots=1, **LN), row * (6 * N + 2 * N)),
    "edge launch, slot order, pair sums": (lambda: ops.tc_mlp_chain(e_slot, layers, gather0=(P, s_src), gather1=(Q, s_dst),
                                                                    residual=e_slot, out=out_n, edge_slots=2, **LN),
                                           row * (4 * N + 3 * N)),
    "node launch, index-driven agg": (lambda: ops.tc_mlp_chain(e, layers, agg=(g.dst_rowptr, g.dst_eid), **node_kw),
                                      row * (E + 3 * N)),
    "node launch, paired operand": (lambda: ops.tc_mlp_chain(e_slot, layers, paired=True, **node_kw), row * (5 * N)),
    "node launch, plain two-operand": (lambda: ops.tc_mlp_chain(agg, layers, **node_kw), row * 4 * N),
}
res = {k: [] for k in cases}
for _ in range(5):
    for name, (fn, nbytes) in cases.items():
        res[name].append(timeit(fn))
print(f"{torch.cuda.get_device_name()}  B={B} graphs of {r}x{r}: N={N} nodes, E={E} edges, {2 * N} slots")
for name, (fn, nbytes) in cases.items():
    med = statistics.median(res[name])
    print(f"{name:36s} median {med:7.3f} ms  (min {min(res[name]):7.3f}, max {max(res[name]):7.3f})  "
          f"{nbytes / med / 1e6:6.0f} GB/s algorithmic")
