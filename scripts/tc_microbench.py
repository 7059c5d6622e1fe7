#!/usr/bin/env python
"""Micro-benchmark of the tcgen05 linear engine per epilogue mode (CUDA events, L2 flushed).

    python scripts/tc_microbench.py [M] [case filter]"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from graphnet_classifier_b200 import ops, build
build.build()

def timeit(fn, n=5):
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(2): fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); fn(); e.record(); torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    return min(ts), sum(ts) / len(ts)

M = int(sys.argv[1]) if len(sys.argv) > 1 else 2_080_768
dev = "cuda"
A = torch.randn(M, 128, device=dev); W = torch.randn(128, 128, device=dev) / 11; b = torch.randn(128, device=dev)
g = torch.ones(128, device=dev); be = torch.zeros(128, device=dev); res = torch.randn(M, 128, device=dev)
R = M // 2
P = torch.randn(R, 128, device=dev); Q = torch.randn(R, 128, device=dev)
i0 = (torch.arange(M, device=dev) // 2).int(); i1 = ((torch.arange(M, device=dev) // 2 + 7) % R).int()
w2 = torch.randn(1, 128, device=dev); b2 = torch.randn(1, device=dev)
out = torch.empty(M, 128, device=dev)
z_out = torch.empty(M, 128, device=dev); mean_out = torch.empty(M, device=dev); rstd_out = torch.empty(M, device=dev)
cases = {
    "plain": lambda: ops.tc_linear(A, W, out=out),
    "bias_relu": lambda: ops.tc_linear(A, W, bias=b, relu=True, out=out),
    "bias_relu_gather2": lambda: ops.tc_linear(A, W, bias=b, relu=True, gather0=(P, i0), gather1=(Q, i1), out=out),
    "layernorm_res": lambda: ops.tc_linear(A, W, bias=b, gamma=g, beta=be, residual=res, out=out),
    "layernorm_res_save": lambda: ops.tc_linear(A, W, bias=b, gamma=g, beta=be, residual=res, out=out,
                                                ln_save=(z_out, mean_out, rstd_out)),
    "relu_dot": lambda: ops.tc_linear(A, W, bias=b, relu=True, dot_w=w2, dot_b=b2),
    "fp32_linear": lambda: ops.linear([A], W, b, relu=True),
    "copy_rw(torch)": lambda: out.copy_(A),
}
filt = sys.argv[2] if len(sys.argv) > 2 else ""
for name, fn in cases.items():
    if filt not in name:
        continue
    best, avg = timeit(fn)
    gb = 4.0 * M * 128 * 2 / 1e9
    print(f"{name:22s} M={M}  best {best:8.3f} ms  avg {avg:8.3f} ms   {2.0*M*128*128/best/1e9:8.1f} TFLOP/s  ~{gb/best*1e3:7.0f} GB/s (A+Y only)")
