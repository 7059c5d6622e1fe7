#!/usr/bin/env python
"""Benchmark of the GraphNet_Classifier hot path on B200 (contract: see the task brief).

    python bench.py --gpus N --steps K --warmup W              # our arm
    python bench.py --impl reference --gpus N --steps K ...    # reference CPU arm
    python bench.py ... --dump-outputs DIR                     # also write the last timed step's logits to DIR

Workload (BASELINE.json configs[1]): GNN inference, resize 128 pixel-grid graphs,
batch 512 synthetic RGB images per GPU (weak scaling).  One "step" = graph build +
GraphNet forward + classifier head for one batch.  ``value`` is graphs/s with the
uint8 images already resident in HBM; ``e2e`` is the same through the public
pipeline call with pinned HOST images (H2D + D2H inside the timed region).
The JSON line also carries: the roofline of the dominant kernel (``traffic`` from an ncu
capture recorded in profiles/kernel_traffic.json, valid only for the profiled sources), the
aggregation kernel's HBM roofline, ``generic_path`` (the same step with the grid shortcuts
off), ``train`` (fwd + bwd + gradient all-reduce + Adam at BASELINE configs[2]'s per-GPU
shape, with its own HBM roofline, the all-reduce timed alone and the oracle's train loop
as CPU baseline), ``configs`` (bounded sub-blocks for BASELINE configs[0], [3] and [4] at
N = 1) and the CPU baseline (the oracle = a validated port of the reference, timed on this
box's host cores).

Only the cpu_baseline leg and ``--impl reference`` import ``oracle/``.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "graphs_per_sec_inference_resize128_batch512_per_gpu"
UNIT = "graphs/s"
FWD_FLOP_PER_NODE = 525_568          # SURVEY.md 8d: fwd FLOPs per graph = 525568*N + 557824*E
FWD_FLOP_PER_EDGE = 557_824


def _count(least: int):
    def integer(s: str) -> int:
        v = int(s)
        if v < least:
            raise argparse.ArgumentTypeError(f"must be >= {least}, got {v}")
        return v
    return integer


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_count(1), default=5, help="timed steps of the headline inference step")
    ap.add_argument("--warmup", type=_count(0), default=3)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed inference step returned in its last step (logits, float32) as "
                         "DIR/logits.npy (DIR/logits_rank<R>.npy per rank when there are several); the inputs are "
                         "seeded, so two builds run with the same arguments can be compared output for output")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--resize", type=int, default=128)
    ap.add_argument("--batch", type=int, default=512, help="graphs per GPU per step")
    ap.add_argument("--train-batch", type=int, default=512, help="graphs per GPU per training step")
    ap.add_argument("--train-steps", type=int, default=10)
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE configs[0]/[3]/[4] sub-blocks (N=1 only)")
    ap.add_argument("--c4-batch", type=int, default=256, help="images of the bounded config-4 (superpixel) sub-block")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-staging", action="store_true")
    ap.add_argument("--no-power", action="store_true", help="skip the board-power block")
    ap.add_argument("--power-seconds", type=float, default=3.0)
    ap.add_argument("--cpu-graphs", type=int, default=256, help="graphs in the bounded CPU sample")
    ap.add_argument("--ref-graphs-per-step", type=int, default=32)
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of our arm's timed step; it does not apply to --impl reference")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], bf16=p["bf16_tflops"], bf16_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    source="MEASURED_PEAKS.json (measured)")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, source="B200_PROFILING.md fallback")


def source_sha(*names) -> str:
    """sha256 (first 16 hex digits) of the named kernel sources: the key under which an ncu capture of a kernel is valid."""
    import hashlib
    h = hashlib.sha256()
    for n in names:
        with open(os.path.join(ROOT, "graphnet_classifier_b200", "csrc", n), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def measured_traffic(key: str, sources):
    """DRAM bytes (read + write) of ONE launch of kernel ``key`` from an ``ncu --set full`` capture recorded in
    profiles/kernel_traffic.json, valid only while the kernel's sources are the ones that were profiled; otherwise
    None - a number copied from an older kernel would be a claim about code that no longer exists."""
    path = os.path.join(ROOT, "profiles", "kernel_traffic.json")
    if not os.path.exists(path):
        return None, None
    with open(path) as f:
        ent = json.load(f).get(key)
    if not ent or ent.get("source_sha") != source_sha(*sources):
        return None, None
    return float(ent["dram_bytes_read"]) + float(ent["dram_bytes_write"]), ent.get("from")


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict, suffix: str = "") -> None:
    """Writes each tensor as ``out_dir/<name><suffix>.npy`` (float64 stays float64, everything else becomes float32)."""
    import numpy as np
    host = {}
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        host[name] = a if a.dtype == np.float64 else a.astype(np.float32)
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit; use a smaller --batch")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int, period_ms: int = 200):
        self.index, self.rows, self.proc, self.thread, self.period_ms = index, [], None, None, int(period_ms)

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", str(self.period_ms), "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                clk, mx = float(r[0]), float(r[1])
            except (ValueError, IndexError):
                continue
            try:
                watts = float(r[2])
            except (ValueError, IndexError):
                watts = None
            sm.append((clk, watts))
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        # "under load" = samples whose board power is within 40 % of the highest seen (the tensor-core kernels of this path
        # run AT the board's power cap, where the SM clock sits below its maximum: selecting by clock would pick the idle
        # samples); without power readings, all samples
        pw = [w for _, w in sm if w is not None]
        busy = [(c, w) for c, w in sm if w is not None and w >= 0.6 * max(pw)] if pw else sm
        clks = sorted(c for c, _ in busy)
        med = clks[len(clks) // 2] if clks else None
        watts = sorted(w for _, w in busy if w is not None)
        return dict(sm_mhz=med, sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm), samples_under_load=len(busy),
                    power_w=watts[len(watts) // 2] if watts else None)


# ------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle (validated port of the reference) on host cores
# ------------------------------------------------------------------------------
def cpu_reference_run(resize: int, n_graphs: int, warm: int, state_dict=None, seed: int = 0):
    """One graph per step exactly like the reference loop (utils/train_model.py:35-45 minus
    the backward): builder (numpy) + loader casts + CombinedModel forward under no_grad."""
    import numpy as np
    import torch
    from oracle import gnn as ognn
    from oracle import graph_build as ogb

    torch.set_num_threads(os.cpu_count() or 1)      # torchrun exports OMP_NUM_THREADS=1
    model = ognn.build_reference_config_model(resize, seed=0)
    if state_dict is not None:
        model.load_state_dict(state_dict)
    model.eval()
    imgs = np.random.default_rng(seed).integers(0, 256, (n_graphs + warm, resize, resize, 3), dtype=np.uint8)
    outs = []
    with torch.no_grad():
        for i in range(warm):
            model(ogb.to_model_inputs(*ogb.pixel_graph(imgs[i])))
        t0 = time.perf_counter()
        for i in range(warm, warm + n_graphs):
            outs.append(model(ogb.to_model_inputs(*ogb.pixel_graph(imgs[i]))))
        dt = time.perf_counter() - t0
    return n_graphs / dt, dt, torch.get_num_threads(), torch.stack(outs), imgs[warm:]


def cpu_train_run(resize: int, n_graphs: int, warm: int = 1):
    """The reference's training loop on the host cores (utils/train_model.py:35-42: one Adam step per graph):
    builder + forward + cross entropy + backward + Adam, oracle port, bounded sample."""
    import numpy as np
    import torch
    from oracle import gnn as ognn
    from oracle import graph_build as ogb

    torch.set_num_threads(os.cpu_count() or 1)
    model = ognn.build_reference_config_model(resize, seed=0)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    rng = np.random.default_rng(7)
    imgs = rng.integers(0, 256, (n_graphs + warm, resize, resize, 3), dtype=np.uint8)
    labs = rng.integers(0, 2, n_graphs + warm)
    t0 = 0.0
    for i in range(n_graphs + warm):
        if i == warm:
            t0 = time.perf_counter()
        loss = torch.nn.functional.cross_entropy(model(ogb.to_model_inputs(*ogb.pixel_graph(imgs[i]))), torch.tensor(int(labs[i])))
        opt.zero_grad(); loss.backward(); opt.step(); loss.item()
    dt = time.perf_counter() - t0
    return {"value": n_graphs / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{n_graphs} graphs of resize {resize}, one optimizer step per graph as the reference loop does "
                      f"(builder + forward + CE + backward + Adam), {dt:.1f} s"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    g = args.ref_graphs_per_step
    # warm-up steps then exactly K timed steps of g graphs each
    import numpy as np
    from oracle import gnn as ognn
    from oracle import graph_build as ogb
    torch.set_num_threads(os.cpu_count() or 1)      # torchrun exports OMP_NUM_THREADS=1
    model = ognn.build_reference_config_model(args.resize, seed=0).eval()
    total = (args.warmup + args.steps) * g
    imgs = np.random.default_rng(0).integers(0, 256, (total, args.resize, args.resize, 3), dtype=np.uint8)
    with torch.no_grad():
        k = 0
        for _ in range(args.warmup):
            for _ in range(g):
                model(ogb.to_model_inputs(*ogb.pixel_graph(imgs[k]))); k += 1
        t0 = time.perf_counter()
        for _ in range(args.steps):
            for _ in range(g):
                model(ogb.to_model_inputs(*ogb.pixel_graph(imgs[k]))); k += 1
        dt = time.perf_counter() - t0
    v = args.steps * g / dt
    cores = torch.get_num_threads()
    sample = f"{g} graphs per step, one graph per forward (reference loop), resize {args.resize}, {cores} threads"
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"GNN inference, resize {args.resize} pixel-grid graphs (BASELINE configs[1]); "
                               f"reference CPU path = oracle port, bounded sample", "resize": args.resize,
                   "graphs_per_step": g},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------
# BASELINE configs[0] / [3] / [4] as bounded sub-blocks (N = 1, rank 0): every config has a driver-visible number
# ------------------------------------------------------------------------------
def run_config_blocks(args, dev, pk, flush):
    import numpy as np
    import torch
    from graphnet_classifier_b200 import _lib, ops
    from graphnet_classifier_b200.models.GNN import CombinedModel, GraphNet
    from graphnet_classifier_b200.ops import GraphIndex
    from graphnet_classifier_b200.pipeline import GraphClassifierPipeline
    from graphnet_classifier_b200.utils.distributed import FlatAdam
    from graphnet_classifier_b200.utils.image_to_graph.batched import build_pixel_graphs, build_superpixel_batch
    from graphnet_classifier_b200.utils.image_to_graph.slic import slic_labels

    def med_ms(fn, n=7, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(n):
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(); fn(); e.record()
            torch.cuda.synchronize()
            ts.append(s.elapsed_time(e))
        return sorted(ts)[len(ts) // 2]

    out = {}
    cfg = dict(num_local_features=3, space_dim=2, out_channels=1, n_blocks=3)

    # ---- configs[0]: resize 64 pixel graphs, batch 32 (the reference's own CPU-runnable case, main.py path) ----
    r1, B1 = 64, 32
    torch.manual_seed(0)
    m1 = CombinedModel(GraphNet(**cfg), num_nodes=r1 * r1, classes=2).to(dev)
    p1 = GraphClassifierPipeline(m1, resize_value=r1)
    rng = np.random.default_rng(5)
    im1 = torch.from_numpy(rng.integers(0, 256, (B1, r1, r1, 3), dtype=np.uint8)).pin_memory()
    lb1 = torch.from_numpy(rng.integers(0, 2, B1)).to(dev)
    im1d = im1.to(dev)
    inf_ms = med_ms(lambda: p1.infer(im1d))
    e2e_ms = med_ms(lambda: p1.infer(im1).cpu())
    c1 = {"what": f"resize {r1} pixel-grid graphs, batch {B1} (BASELINE configs[0])",
          "inference": {"value": B1 / inf_ms * 1e3, "unit": UNIT, "ms_per_step": inf_ms},
          "e2e": {"value": B1 / e2e_ms * 1e3, "unit": UNIT, "ms_per_step": e2e_ms,
                  "h2d_bytes_per_step": int(im1.numel()), "d2h_bytes_per_step": B1 * 8}}
    try:        # the same batch through the captured CUDA graph (GraphClassifierPipeline.infer_graphed): this size is launch-bound
        g_ms = med_ms(lambda: p1.infer_graphed(im1d))
        same = bool(torch.equal(p1.infer_graphed(im1d), p1.infer(im1d)))
        c1["inference_graphed"] = {"value": B1 / g_ms * 1e3, "unit": UNIT, "ms_per_step": g_ms, "equal_to_infer": same}
    except Exception as ex:
        c1["inference_graphed"] = {"error": repr(ex)}
    if not args.no_cpu_baseline:
        sd = {k: v.detach().cpu() for k, v in m1.state_dict().items()}
        v, dt, cores, ref_logits, ref_imgs = cpu_reference_run(r1, B1, 1, state_dict=sd, seed=99)
        got = p1.infer(torch.from_numpy(ref_imgs)).cpu()
        c1["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                              "sample": f"{B1} graphs, one per forward (reference loop), {dt:.1f} s",
                              "max_rel_logit_diff_vs_gpu": float((got - ref_logits).abs().max() / ref_logits.abs().max())}
    opt1 = FlatAdam(m1.parameters(), lr=1e-3)
    tr_ms = med_ms(lambda: p1.train_step(im1d, lb1, opt1), n=5, warm=3)
    c1["train"] = {"value": B1 / tr_ms * 1e3, "unit": UNIT, "ms_per_step": tr_ms,
                   "what": "one optimizer step on the 32-graph batch (build + forward + CE + backward + Adam)"}
    if not args.no_cpu_baseline:
        c1["train"]["cpu_baseline"] = cpu_train_run(r1, 8)
    out["c1_resize64_batch32"] = c1
    del m1, p1, opt1

    # ---- configs[3]: superpixel graph build + GNN at resize 256 (bounded batch) ----
    r4, B4 = 256, args.c4_batch
    torch.manual_seed(0)
    m4 = CombinedModel(GraphNet(**cfg), num_nodes=r4 // 2, classes=2).to(dev).eval()      # main.py:65-66
    g = torch.Generator(device=dev).manual_seed(0)
    low = torch.rand(B4, 3, 8, 8, device=dev, generator=g)
    im4 = torch.nn.functional.interpolate(low, size=(r4, r4), mode="bilinear", align_corners=False)
    im4 = (im4 + 0.05 * torch.randn(B4, 3, r4, r4, device=dev, generator=g)).clamp(0, 1).mul(255).byte()
    im4 = im4.permute(0, 2, 3, 1).contiguous()
    holder = {}

    def c4_slic():
        holder["labels"] = slic_labels(im4, n_segments=100, compactness=10.0)

    def c4_build():
        holder["gb"] = build_superpixel_batch(im4, labels=holder["labels"], max_nodes=128)

    @torch.no_grad()
    def c4_model():
        holder["logits"] = m4(holder["gb"].as_tuple())

    def c4_all():
        c4_slic(); c4_build(); c4_model()

    t_slic = med_ms(c4_slic, n=5, warm=2)
    t_build = med_ms(c4_build, n=5, warm=2)
    t_model = med_ms(c4_model, n=5, warm=2)
    t_all = med_ms(c4_all, n=5, warm=1)
    gb4 = holder["gb"]
    out["c4_superpixel_resize256"] = {
        "what": f"{B4} synthetic images (smooth blobs + noise) at resize {r4}: device SLIC (100 segments, 10 iterations, "
                f"connectivity enforced) -> superpixel graphs -> block-diagonal batch + CSR -> GraphNet -> pad/truncate "
                f"readout -> head (BASELINE configs[3], bounded batch: {B4} of 1024)",
        "value": B4 / t_all * 1e3, "unit": "images/s", "ms_per_step": t_all,
        "stages_ms": {"slic": t_slic, "graph_build_compaction_csr": t_build, "graphnet_readout_head": t_model},
        "nodes_per_image": gb4.x.shape[0] / B4, "edges_per_image": gb4.edge_index.shape[1] / B4,
        "logits_finite": bool(torch.isfinite(holder["logits"]).all()), "logits_shape": list(holder["logits"].shape),
        "parity": "label map -> graph and the readout are oracle-checked in tests/; SLIC itself is parity-unpinned "
                  "(scikit-image is not vendored by the reference)"}
    del m4, im4, holder, gb4

    # ---- configs[4]: aggregation micro-benchmark against torch index_add_ (bounded rows of the sweep) ----
    rows = []
    for kind, E_t, D in (("grid", 10_000_000, 128), ("random", 10_000_000, 128), ("random", 1_000_000, 32)):
        if kind == "grid":
            Bg = max(1, round(E_t / (2 * 128 * 127)))
            gr = build_pixel_graphs(torch.zeros(Bg, 128, 128, 3, dtype=torch.uint8, device=dev), use_cache=False).graph
        else:
            Nn = E_t // 2
            gg = torch.Generator(device=dev).manual_seed(0)
            ei = torch.stack([torch.randint(0, Nn, (E_t,), device=dev, generator=gg),
                              torch.randint(0, Nn, (E_t,), device=dev, generator=gg)])
            gr = GraphIndex.from_edge_index(ei, Nn, validate=False)
        En, Nn = gr.num_edges, gr.num_nodes
        srcm = torch.randn(En, D, device=dev)
        ms = med_ms(lambda: ops.aggregate(srcm, gr), n=7, warm=3)
        idx = gr.dst.long()
        ref = torch.zeros(Nn, D, device=dev)
        ms_t = med_ms(lambda: ref.zero_().index_add_(0, idx, srcm), n=5, warm=2)
        nbytes = 4.0 * (En * D + En + (Nn + 1) + Nn * D)
        rows.append({"topology": kind, "edges": En, "nodes": Nn, "D": D, "ms": ms, "achieved": nbytes / ms / 1e6,
                     "unit": "GB/s", "peak": pk["hbm"], "frac": nbytes / ms / 1e6 / pk["hbm"],
                     "torch_index_add_ms": ms_t, "speedup_vs_torch_index_add": ms_t / ms})
        del srcm, ref, gr
    out["c5_aggregation"] = {"what": "gnc_agg_csr_sum_f32 (ordered CSR segmented sum, bit-identical to the CPU index_add_) vs "
                                     "torch index_add_ (atomics) on this GPU; bytes = 4(E D + E + N + 1 + N D); the full sweep "
                                     "and the multi-GPU rows are in profiles/ (scripts/agg_sweep*.py)", "rows": rows}
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (our arm) needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world

    from graphnet_classifier_b200 import _lib, ops
    _lib.load()         # the library build() made; the benchmark never compiles, so it runs from a read-only tree
    from graphnet_classifier_b200.models.GNN import CombinedModel, GraphNet
    from graphnet_classifier_b200.pipeline import GraphClassifierPipeline
    from graphnet_classifier_b200.utils.distributed import GradBucket, broadcast_parameters

    r, B = args.resize, args.batch
    N, E = r * r, 2 * r * (r - 1)
    torch.manual_seed(0)
    model = CombinedModel(GraphNet(num_local_features=3, space_dim=2, out_channels=1, n_blocks=3), num_nodes=N,
                          classes=2).to(dev)
    broadcast_parameters(model)
    pipe = GraphClassifierPipeline(model, resize_value=r)
    rng = np.random.default_rng(rank)
    imgs_host = torch.from_numpy(rng.integers(0, 256, (B, r, r, 3), dtype=np.uint8)).pin_memory()
    labels_host = torch.from_numpy(rng.integers(0, 2, B)).pin_memory()
    imgs_dev = imgs_host.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(step_fn, steps, warmup):
        """W untimed steps, then exactly K steps, each bracketed by CUDA events on the
        launching stream, L2 flushed between steps (outside the event pairs)."""
        for _ in range(warmup):
            step_fn()
        barrier()
        evs = []
        wall0 = time.perf_counter()
        for _ in range(steps):
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            step_fn()
            e.record()
            evs.append((s, e))
        barrier()
        wall = time.perf_counter() - wall0
        ms = sum(s.elapsed_time(e) for s, e in evs)
        return max_over_ranks(ms), wall

    # ---- inference, inputs resident in HBM (value) -------------------------------
    last = {}

    def infer_step():
        last["logits"] = pipe.infer(imgs_dev)
        return last["logits"]

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    _lib.reset_launch_count()
    for _ in range(args.warmup):
        infer_step()
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() // max(args.warmup, 1)
    ms_total, wall = timed(infer_step, args.steps, 0)
    clocks = sampler.stop() if rank == 0 else None
    value = n_gpus * B * args.steps / (ms_total / 1e3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logits": last["logits"]}, f"_rank{rank}" if world > 1 else "")

    # ---- board power under this step (outside every timed region) ---------------------------------------------------
    # The tensor-core launches of the path run AT the board's power cap (DESIGN.md section 5): the same step back to back
    # for a few seconds, power and SM clock sampled every 50 ms, next to the enforced limit.
    power = None
    if rank == 0 and not args.no_power:
        try:
            ps = ClockSampler(local_rank, period_ms=50)
            ps.start()
            t0 = time.perf_counter()
            n_pw = 0
            while time.perf_counter() - t0 < args.power_seconds:
                infer_step()
                n_pw += 1
                if n_pw % 4 == 0:
                    torch.cuda.synchronize()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            pw = ps.stop()
            lim = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", str(local_rank)],
                                 capture_output=True, text=True).stdout.strip()
            try:
                lim = float(lim)
            except ValueError:
                lim = None
            power = {"board_w_under_load": pw.get("power_w"), "limit_w": lim, "sm_mhz_under_load": pw.get("sm_mhz"),
                     "sm_max_mhz": pw.get("sm_max_mhz"), "reasons": pw.get("reasons"), "samples_under_load": pw.get("samples_under_load"),
                     "at_power_cap": (pw.get("power_w") is not None and lim is not None and pw["power_w"] >= 0.95 * lim),
                     "steps": n_pw, "seconds": dt, "graphs_per_s_sustained": B * n_pw / dt,
                     "what": "the inference step back to back (no L2 flush, no per-step events), nvidia-smi every 50 ms"}
        except Exception as ex:           # a secondary block never fails the line
            power = {"error": repr(ex)}

    # ---- end to end: pinned host images in, logits back on the host -----------------
    def e2e_step():
        return pipe.infer(imgs_host).cpu()

    e2e_ms, _ = timed(e2e_step, args.steps, 1)
    e2e_value = n_gpus * B * args.steps / (e2e_ms / 1e3)

    # ---- the same step without the grid shortcuts: `pos` is a copy, so the model cannot assume our builder's grid
    # (per-edge geometry + edge encoder on all E rows, block 0 in the generic chained form) ---
    from graphnet_classifier_b200.utils.image_to_graph.batched import build_pixel_graphs

    @torch.no_grad()
    def generic_step():
        outs = []
        mbg = pipe._even_chunk(B, pipe.micro_batch)
        for lo in range(0, B, mbg):
            gb = build_pixel_graphs(imgs_dev[lo:lo + mbg])
            outs.append(model((gb.x, gb.pos.clone(), gb.edge_index)))
        return outs

    _lib.reset_launch_count()
    generic_step()
    torch.cuda.synchronize()
    g_launches = _lib.launch_count()
    g_steps = max(3, args.steps // 2)
    g_ms, _ = timed(generic_step, g_steps, 1)
    generic = {"value": n_gpus * B * g_steps / (g_ms / 1e3), "unit": UNIT, "ms_per_step": g_ms / g_steps, "steps": g_steps,
               "gpu_launches_per_step": g_launches,
               "what": "same workload with a cloned `pos` tensor: arbitrary-topology path (edge geometry kernel, edge "
                       "encoder on all E rows, no edge-class tables), CSR still the builder's"}

    # ---- per-kernel attribution of one inference step (events around every launch) ---
    ops.PROFILE = ops.KernelProfile()
    infer_step()
    prof = ops.PROFILE.summary()
    ops.PROFILE = None
    prof_ms = sum(d["ms"] for d in prof.values())
    pk = peaks()
    fp32_fma_peak = 148 * 128 * 2 * 1.965e9 / 1e12
    dom_name = max(prof, key=lambda k: prof[k]["ms"])
    dom = prof[dom_name]
    dom_s = dom["ms"] / 1e3
    if dom_name == "tc_linear":
        # one [rows,128] x [128,128] layer per launch: 32 fp32-FLOP per byte of unavoidable traffic,
        # i.e. HBM-bound even at 3 tensor-core passes per product (DESIGN.md section 4)
        gbs = dom["bytes"] / dom_s / 1e9
        roofline = {
            "kernel": "tc_linear_kernel (tcgen05 kind::tf32, 3xTF32 split, TMEM accumulators)", "bound": "hbm",
            "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"], "traffic": None,
            "peak_source": pk["source"],
            "algorithmic_bytes_per_step": dom["bytes"], "launches_per_step": dom["calls"],
            "avg_launch_ms": dom["ms"] / dom["calls"], "share_of_step": dom["ms"] / prof_ms if prof_ms else None,
            "fp32_equivalent_tflops": dom["flops"] / dom_s / 1e12,
            "tensor_tflops_executed": 3.0 * dom["flops"] / dom_s / 1e12,
            "tensor_frac_of_bf16_sustained": 3.0 * dom["flops"] / dom_s / 1e12 / pk["bf16_sustained"],
            "note": "bytes = every operand/result row once per launch, summed over the step's launches; "
                    "time = CUDA events around each launch on the launching stream",
        }
    elif dom_name == "tc_mlp_chain":
        # a whole 2-3 layer MLP per launch, hidden activations on chip: 64-96 fp32-FLOP per byte of
        # unavoidable traffic and three fp16 tensor-core passes per product -> bound by the tensor pipe
        tf = 3.0 * dom["flops"] / dom_s / 1e12
        gbs = dom["bytes"] / dom_s / 1e9
        traffic_edge, traffic_from = measured_traffic(f"tc_chain2_edge_b{B}_r{r}", ("tc_chain.cu", "common.cuh"))
        roofline = {
            "kernel": "tc_chain_kernel (tcgen05 kind::f16 cta_group::2, two-piece fp16 split, 3 MMAs per product, "
                      "hidden activations in TMEM)", "bound": "tensor",
            "achieved": tf, "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": tf / pk["bf16_sustained"],
            # DRAM bytes of the largest launch of this kernel family at this workload (edge processor, 16.6 M rows,
            # tc_chain2_kernel<1>): dram__bytes_read + dram__bytes_write of one ncu --set full capture, looked up by
            # the hash of the kernel's sources (null when the kernel has changed since the capture)
            "traffic": traffic_edge,
            "traffic_from": traffic_from,
            "traffic_algorithmic_bytes_same_launch": 4.0 * 128 * (2 * B * E + 2 * B * N),
            "peak_source": pk["source"] + ": dense bf16 cuBLAS, sustained (kernel timed inside a long step)",
            "executed_tensor_flops_per_step": 3.0 * dom["flops"], "fp32_equivalent_tflops": dom["flops"] / dom_s / 1e12,
            "launches_per_step": dom["calls"], "avg_launch_ms": dom["ms"] / dom["calls"],
            "share_of_step": dom["ms"] / prof_ms if prof_ms else None,
            "hbm_algorithmic_gbs": gbs, "hbm_frac": gbs / pk["hbm"], "algorithmic_bytes_per_step": dom["bytes"],
            "note": "achieved = executed tensor FLOPs (3 fp16 MMAs per fp32-accurate product) / CUDA-event time of "
                    "the launches; hbm_* = every operand/result row once per launch over the same time",
        }
    else:
        tf = dom["flops"] / dom_s / 1e12 if dom_s > 0 else 0.0
        roofline = {
            "kernel": f"{dom_name} (sgemm_128x128_kernel, fp32 FMA)", "bound": "tensor",
            "achieved": tf, "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": tf / pk["bf16_sustained"],
            "traffic": None,
            "peak_source": pk["source"] + ": dense bf16 cuBLAS, sustained (kernel timed inside a long step)",
            "note": "fp32 CUDA-core GEMM (1e-5 parity rules out single-pass TF32/BF16); "
                    f"fraction of the nominal fp32 FMA peak ({fp32_fma_peak:.1f} TFLOP/s) = {tf / fp32_fma_peak:.3f}",
            "launches_per_step": dom["calls"], "share_of_step": dom["ms"] / prof_ms if prof_ms else None,
            "algorithmic_flops_per_step": dom["flops"],
        }
    kernel_shares = {k: {"ms": round(d["ms"], 3), "calls": d["calls"], "share": round(d["ms"] / prof_ms, 4)}
                     for k, d in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}

    # ---- aggregation kernel alone at the step's shape (HBM roofline, BASELINE metric) ---
    mb = min(B, pipe.micro_batch)
    gb = build_pixel_graphs(imgs_dev[:mb])
    e_lat = torch.randn(gb.graph.num_edges, 128, device=dev)
    for _ in range(3):
        ops.aggregate(e_lat, gb.graph)
    torch.cuda.synchronize()
    agg_ms = []
    for _ in range(10):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); ops.aggregate(e_lat, gb.graph); e.record()
        torch.cuda.synchronize()
        agg_ms.append(s.elapsed_time(e))
    agg_ms = sum(agg_ms) / len(agg_ms)
    En, Nn = gb.graph.num_edges, gb.graph.num_nodes
    agg_bytes = 4.0 * (En * 128 + En + (Nn + 1) + Nn * 128)
    agg_gbs = agg_bytes / (agg_ms / 1e3) / 1e9
    roofline_agg = {"kernel": "agg_csr_sum_vec_kernel<32,1>", "bound": "hbm", "achieved": agg_gbs, "peak": pk["hbm"],
                    "unit": "GB/s", "frac": agg_gbs / pk["hbm"], "traffic": None, "edges": En, "nodes": Nn, "D": 128,
                    "algorithmic_bytes_per_launch": agg_bytes, "ms_per_launch": agg_ms, "peak_source": pk["source"],
                    "note": "the kernel timed alone at the step's shape: training and graphs with in-degree > 2 launch it; the "
                            "inference step on grid graphs folds this sum into the node processor's launch "
                            "(tc_mlp_chain agg=..., GNC_FUSE_AGG=0 restores the launch)"}
    del e_lat, gb

    # ---- training: fwd + bwd + gradient all-reduce + Adam (BASELINE configs[2] per-GPU shape) ---
    train = None
    if not args.no_train and args.train_steps > 0:
        from graphnet_classifier_b200.utils.distributed import FlatAdam
        Bt = args.train_batch
        timg = imgs_dev[:Bt] if Bt <= B else torch.from_numpy(rng.integers(0, 256, (Bt, r, r, 3), dtype=np.uint8)).to(dev)
        tlab = torch.from_numpy(rng.integers(0, 2, Bt)).to(dev)
        opt = FlatAdam(model.parameters(), lr=1e-3)         # flat parameters + gradients: bucket and optimizer in one

        def train_step():
            return pipe.train_step(timg, tlab, opt)

        _lib.reset_launch_count()
        for _ in range(2):
            train_step()
        torch.cuda.synchronize()
        t_launches = _lib.launch_count() // 2
        t_ms, _ = timed(train_step, args.train_steps, 0)
        # the one collective of the path, timed alone on the same bucket (NCCL all-reduce of the flat gradient buffer)
        ar_ms = None
        if world > 1:
            ar = []
            for _ in range(3):
                opt.all_reduce(average=True)
            barrier()
            for _ in range(10):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record(); opt.all_reduce(average=True); e.record()
                torch.cuda.synchronize()
                ar.append(s.elapsed_time(e))
            ar_ms = max_over_ranks(sorted(ar)[len(ar) // 2])
        # per-kernel attribution of one training step: the step is a sequence of HBM-bound passes, so its roofline is
        # algorithmic bytes moved / time against the measured copy bandwidth
        ops.PROFILE = ops.KernelProfile()
        train_step()
        tprof = ops.PROFILE.summary()
        ops.PROFILE = None
        tp_ms = sum(d["ms"] for d in tprof.values())
        tp_bytes = sum(d["bytes"] for d in tprof.values())
        t_gbs = tp_bytes / (tp_ms / 1e3) / 1e9 if tp_ms else 0.0
        tdom = max(tprof, key=lambda k: tprof[k]["ms"])
        train = {"value": n_gpus * Bt * args.train_steps / (t_ms / 1e3), "unit": UNIT, "steps": args.train_steps,
                 "ms_per_step": t_ms / args.train_steps, "graphs_per_gpu_per_step": Bt,
                 "micro_batch": pipe.train_micro_batch, "gpu_launches_per_step": t_launches,
                 "allreduce_ms": ar_ms, "allreduce_bytes": int(opt.flat.numel() * 4),
                 "optimizer": "FlatAdam (one launch over the flat parameter / gradient buffers)",
                 "roofline": {"bound": "hbm", "achieved": t_gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": t_gbs / pk["hbm"],
                              "traffic": None, "algorithmic_bytes_per_step": tp_bytes, "profiled_kernel_ms": tp_ms,
                              "dominant_kernel": tdom,
                              "dominant_kernel_gbs": tprof[tdom]["bytes"] / (tprof[tdom]["ms"] / 1e3) / 1e9,
                              "note": "all launches of one step: every operand / result row once per launch, CUDA events "
                                      "around each launch"},
                 "kernel_shares": {k: {"ms": round(d["ms"], 3), "calls": d["calls"],
                                       "gbs": round(d["bytes"] / max(d["ms"], 1e-9) / 1e6, 1)}
                                   for k, d in sorted(tprof.items(), key=lambda kv: -kv[1]["ms"])[:8]},
                 "what": "graph build + forward + CE + backward + flat-bucket all-reduce (NCCL) + Adam"}
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            train["cpu_baseline"] = cpu_train_run(r, 6)
        del opt

    # ---- CPU baseline (rank 0, N=1 only): oracle port on this box's host cores -----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
        v, dt, cores, ref_logits, ref_imgs = cpu_reference_run(r, args.cpu_graphs, 1, state_dict=sd, seed=1234)
        # parity gate on the very graphs the CPU just classified
        got = pipe.infer(torch.from_numpy(ref_imgs)).cpu()
        err = float((got - ref_logits).abs().max() / ref_logits.abs().max())
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{args.cpu_graphs} graphs of the same workload (resize {r}), one graph per forward as the "
                         f"reference loop does, builder included, {dt:.1f} s",
               "host_cpu_count": os.cpu_count(), "max_rel_logit_diff_vs_gpu": err}

    # ---- input staging (SURVEY.md 8f rank 1): unresized photos -> Pillow-exact device resize -> same path ---
    staging = None
    if not args.no_staging:
        ph, pw = 375, 500
        photos_host = torch.from_numpy(rng.integers(0, 256, (B, ph, pw, 3), dtype=np.uint8)).pin_memory()
        photos_dev = photos_host.to(dev)
        rs_ms, _ = timed(lambda: ops.resize_bicubic(photos_dev, r, r), args.steps, 2)
        ph_ms, _ = timed(lambda: pipe.infer(photos_host).cpu(), args.steps, 1)
        rs_bytes = 3.0 * B * (ph * pw + r * r)
        rs_gbs = rs_bytes * args.steps / (rs_ms / 1e3) / 1e9
        staging = {
            "what": f"{B} RGB photos {ph}x{pw} per GPU -> resize {r} (Pillow BICUBIC, bit-exact) on the device",
            "resize_images_per_s": n_gpus * B * args.steps / (rs_ms / 1e3), "resize_ms_per_step": rs_ms / args.steps,
            "roofline": {"kernel": "resize_h_reg_kernel + resize_v_kernel", "bound": "hbm", "achieved": rs_gbs,
                         "peak": peaks()["hbm"], "unit": "GB/s", "frac": rs_gbs / peaks()["hbm"], "traffic": None,
                         "algorithmic_bytes_per_step": rs_bytes,
                         "note": "bytes = photo in + resized image out; the kernels are bound by integer multiply-add issue"},
            "e2e_from_photos": {"value": n_gpus * B * args.steps / (ph_ms / 1e3), "unit": UNIT,
                                "h2d_bytes_per_step": int(photos_host.numel()), "d2h_bytes_per_step": int(B * 2 * 4),
                                "ms_per_step": ph_ms / args.steps,
                                "api": "GraphClassifierPipeline.infer(pinned uint8 host photos) -> logits.cpu()"},
        }
        del photos_dev, photos_host
        # ---- from image FILES: threaded host decode (utils/staging.DecodePool) -> pinned double-buffered copies -> the
        # same device path.  The files are synthetic JPEGs written to a temporary directory (no dataset on the box).
        if world == 1:      # the host cores are shared by the ranks of a box: measured where one rank has them all
            import shutil
            import tempfile
            from PIL import Image
            from graphnet_classifier_b200.utils.staging import DecodePool, infer_files
            n_files = B
            tmpd = tempfile.mkdtemp(prefix="gnc_bench_")
            try:
                paths = []
                for i in range(n_files):
                    low = rng.integers(0, 256, (ph // 16 + 2, pw // 16 + 2, 3), dtype=np.uint8)
                    im = Image.fromarray(low).resize((pw, ph), Image.BICUBIC)
                    pth = os.path.join(tmpd, f"{i}.jpg")
                    im.save(pth, quality=90)
                    paths.append(pth)
                file_bytes = sum(os.path.getsize(pth) for pth in paths)
                t0 = time.perf_counter()
                for pth in paths[:32]:
                    np.asarray(Image.open(pth).convert("RGB"))
                one_core = 32 / (time.perf_counter() - t0)
                with DecodePool(device=dev, device_jpeg=True) as pool:
                    infer_files(pipe, paths, pool=pool).cpu()                # warm-up: staging buffers, resize tables
                    torch.cuda.synchronize()
                    reps = 3
                    t0 = time.perf_counter()
                    for _ in range(reps):
                        infer_files(pipe, paths, pool=pool).cpu()
                    torch.cuda.synchronize()
                    dt = (time.perf_counter() - t0) / reps
                    workers, pool_stats = pool.workers, dict(pool.stats)
                # the device JPEG decoder alone (csrc/jpeg.cu): file bytes already in host memory -> RGB pixels in HBM
                from graphnet_classifier_b200.utils import jpeg as gjpeg
                datas = [open(pth, "rb").read() for pth in paths]
                jst = {}
                for _ in range(2):
                    gjpeg.decode_batch(datas, dev, staging=jst)
                torch.cuda.synchronize()
                jms = []
                for _ in range(5):
                    s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    s_.record(); gjpeg.decode_batch(datas, dev, staging=jst); e_.record()
                    torch.cuda.synchronize()
                    jms.append(s_.elapsed_time(e_))
                jms = sorted(jms)[2]
                with DecodePool(device=dev, device_jpeg=False) as pool:   # the host-decode form of the same call
                    infer_files(pipe, paths, pool=pool).cpu()
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for _ in range(reps):
                        infer_files(pipe, paths, pool=pool).cpu()
                    torch.cuda.synchronize()
                    dt_host = (time.perf_counter() - t0) / reps
                probe = DecodePool(device=dev)
                auto_is_device = probe.device_jpeg
                probe.close()
                dt_auto = dt if auto_is_device else dt_host
                staging["e2e_from_files"] = {
                    "value": n_files / dt_auto, "unit": UNIT, "files_per_step": n_files, "ms_per_step": dt_auto * 1e3,
                    "default_decoder": "device" if auto_is_device else "host processes",
                    "default_rule": "baseline JPEG files are decoded on the device, everything else by Pillow on worker processes",
                    "device_decode_form": {
                        "value": n_files / dt, "unit": UNIT, "ms_per_step": dt * 1e3, "files_by_decoder": pool_stats,
                        "h2d_bytes_per_step": file_bytes,
                        "what": "csrc/jpeg.cu: Huffman + IDCT + upsampling + colour on the GPU, bit-identical to Pillow; the "
                                "pool's threads only read and parse the files; only the compressed bytes cross PCIe"},
                    "host_decode_form": {
                        "value": n_files / dt_host, "unit": UNIT, "ms_per_step": dt_host * 1e3,
                        "h2d_bytes_per_step": n_files * ph * pw * 3,
                        "what": "Pillow on worker processes into shared pinned memory, double-buffered copies"},
                    "device_jpeg_decode": {
                        "images_per_s": n_files / (jms / 1e3), "ms_per_step": jms,
                        "what": "gnc_jpeg_decode_rgb_u8 alone on the files' bytes (host -> device copy of the compressed "
                                "bytes included), CUDA events"},
                    "decode_workers": workers, "host_cpu_count": os.cpu_count(),
                    "one_thread_pil_decode_images_per_s": one_core, "file_bytes_per_step": file_bytes,
                    "h2d_bytes_per_step": file_bytes if auto_is_device else n_files * ph * pw * 3,
                    "d2h_bytes_per_step": n_files * 8,
                    "timing": "wall clock around the whole call (host work is part of it), this rank only",
                    "api": "utils.staging.infer_files(pipeline, jpeg paths) -> logits.cpu(): decode (device or host "
                           "processes) -> Pillow-exact device resize -> graph build -> GraphNet"}
                # nvJPEG (library: torchvision.io.decode_jpeg on the device) on the same files, measured as the
                # alternative to the host decode.  NOT on the default path: its IDCT / chroma upsampling differ from
                # libjpeg's, so the pixels are not the reference's - the difference against PIL is stated here.
                try:
                    from torchvision.io import decode_jpeg, read_file
                    datas = [read_file(pth) for pth in paths]
                    for _ in range(2):
                        dec = decode_jpeg(datas, device=dev)
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for _ in range(3):
                        dec = decode_jpeg(datas, device=dev)
                    torch.cuda.synchronize()
                    nv_dt = (time.perf_counter() - t0) / 3
                    worst, mean, same = 0, 0.0, 0
                    for pth, dimg in list(zip(paths, dec))[:64]:
                        ref_px = torch.from_numpy(np.array(Image.open(pth).convert("RGB"))).to(dev)
                        diff = (dimg.permute(1, 2, 0).int() - ref_px.int()).abs()
                        worst = max(worst, int(diff.max()))
                        mean += float(diff.float().mean()) / 64
                        same += int(diff.max() == 0)
                    staging["nvjpeg_alternative"] = {
                        "images_per_s": n_files / nv_dt, "ms_per_step": nv_dt * 1e3, "files_per_step": n_files,
                        "max_abs_pixel_diff_vs_pil": worst, "mean_abs_pixel_diff_vs_pil": mean,
                        "bit_identical_images_of_64": same,
                        "what": "torchvision.io.decode_jpeg(list of file bytes, device=cuda) = nvJPEG batched decode (file "
                                "bytes already in host memory); library call, reported for comparison only"}
                    del dec, datas
                except Exception as exc:            # torchvision built without nvJPEG, or absent
                    staging["nvjpeg_alternative"] = {"unavailable": str(exc)[:200]}
            except Exception as exc:                # a secondary block must never cost the headline line
                staging["e2e_from_files"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
            finally:
                shutil.rmtree(tmpd, ignore_errors=True)

    configs = None
    if rank == 0 and world == 1 and not args.no_configs:
        torch.cuda.empty_cache()
        try:
            configs = run_config_blocks(args, dev, pk, flush)
        except Exception as exc:                    # a secondary block must never cost the headline line
            configs = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"GNN inference, resize {r} pixel-grid graphs, batch {B} per GPU "
                                   f"(BASELINE configs[1]); graph build + GraphNet(3 blocks, width 128) + head",
                       "resize": r, "graphs_per_gpu": B, "nodes_per_graph": N, "edges_per_graph": E,
                       "dense_engine": ops.ENGINE, "micro_batch": pipe.micro_batch, "parallelism": f"dp{n_gpus} (independent graphs, no data-path collective)",
                       "l2": "256 MiB buffer zeroed between timed steps (outside the event pairs); "
                             "per-step working set (8.5 GB edge tensors) >> 126 MB L2",
                       "algorithmic_fwd_tflop_per_step": B * (FWD_FLOP_PER_NODE * N + FWD_FLOP_PER_EDGE * E) / 1e12},
            "wall_s_timed_region": wall,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(imgs_host.numel()),
                    "d2h_bytes_per_step": int(B * 2 * 4), "ms_per_step": e2e_ms / args.steps,
                    "api": "GraphClassifierPipeline.infer(pinned uint8 host images) -> logits.cpu()"},
            "gpu_launches": int(launches_per_step * args.steps),
            "gpu_launches_per_step": int(launches_per_step),
            "clocks": clocks,
            "power": power,
            "roofline": roofline,
            "roofline_aggregation": roofline_agg,
            "kernel_shares": kernel_shares,
            "generic_path": generic,
            "train": train,
            "configs": configs,
            "staging": staging,
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
