#!/usr/bin/env python
"""Device PNG decoder (csrc/png.cu) against Pillow on host processes: photo-like PNGs saved by Pillow (smooth gradients
plus noise), checked bit for bit against Pillow, CUDA events, medians of interleaved rounds, with the GPU's name and
power limit from the same run.

    png_bench.py [B] [--out FILE]

Reports: decode_batch wall and kernel time on B files of 375 x 500 and on B files of mixed sizes; DecodePool.stage at
resize 128 with device_png=True against host processes at 15 and at 2 workers (one GPU's share of a 16-core, 8-GPU
box); infer_files end to end in the same three forms; the single-stream rate (MB/s of raw filtered output) of one file
near the raw-size cap decoded alone, which bounds a batch's time from below; and, in a torch.profiler run of its own,
the time of each of the two kernels (inflate, unfilter + convert) on the 375 x 500 batch and on the single file."""
import io, os, subprocess, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from PIL import Image
from graphnet_classifier_b200 import build, ops

LINES = []


def say(s):
    print(s, flush=True)
    LINES.append(s)


def photo(rng, h, w):
    yy, xx = np.mgrid[0:h, 0:w]
    base = np.stack([(xx * 255 // w + yy // 2) % 256, (yy * 255 // h) % 256, ((xx + yy) // 3) % 256], -1)
    px = np.clip(base + rng.integers(-8, 9, (h, w, 3)), 0, 255).astype(np.uint8)
    buf = io.BytesIO()
    Image.fromarray(px).save(buf, format="PNG")
    return buf.getvalue()


def pillow(d):
    return np.asarray(Image.open(io.BytesIO(d)).convert("RGB"))


def median(xs):
    return sorted(xs)[len(xs) // 2]


def decode_bench(name, datas, rounds=7):
    from graphnet_classifier_b200.utils.png import decode_batch
    st = {}
    out = decode_batch(datas, staging=st)
    for d, t in zip(datas, out):
        assert t is not None and np.array_equal(t.cpu().numpy(), pillow(d))
    walls, kernels = [], []
    for _ in range(rounds):
        torch.cuda.synchronize()
        t0 = time.perf_counter(); decode_batch(datas, staging=st); torch.cuda.synchronize()
        walls.append((time.perf_counter() - t0) * 1e3)
        ops.PROFILE = ops.KernelProfile()
        decode_batch(datas, staging=st); torch.cuda.synchronize()
        p = ops.PROFILE.summary()["png_decode"]
        ops.PROFILE = None
        kernels.append(p["ms"] / p["calls"])
    B = len(datas)
    w, k = median(walls), median(kernels)
    say(f"{name}: {B} files, {sum(map(len, datas)) / B / 1e3:.1f} KB each on average, all bit-identical to Pillow: "
        f"decode_batch {w:.2f} ms ({B / w * 1e3:,.0f} files/s), kernels {k:.2f} ms ({B / k * 1e3:,.0f} files/s)")


def write_files(tmp, datas, tag):
    paths = []
    for i, d in enumerate(datas):
        p = os.path.join(tmp, f"{tag}{i}.png")
        with open(p, "wb") as f:
            f.write(d)
        paths.append(p)
    return paths


def pool_bench(paths, rounds=5, r=128):
    from graphnet_classifier_b200.utils.staging import DecodePool, infer_files
    from graphnet_classifier_b200.models.GNN import CombinedModel, GraphNet
    from graphnet_classifier_b200.pipeline import GraphClassifierPipeline
    torch.manual_seed(0)
    model = CombinedModel(GraphNet(num_local_features=3, space_dim=2, out_channels=1, n_blocks=3), num_nodes=r * r).cuda().eval()
    pipe = GraphClassifierPipeline(model, resize_value=r)
    pools = {"device_png": DecodePool(device_png=True), "host 15 processes": DecodePool(workers=15, device_jpeg=False),
             "host 2 processes": DecodePool(workers=2, device_jpeg=False)}
    ref = pools["host 15 processes"].stage(paths, r)
    logits = {}
    for k, pool in pools.items():
        assert torch.equal(pool.stage(paths, r), ref), k
        logits[k] = infer_files(pipe, paths, pool=pool)
    assert all(torch.equal(v, logits["host 15 processes"]) for v in logits.values())
    st = {k: [] for k in pools}
    inf = {k: [] for k in pools}
    for _ in range(rounds):
        for k, pool in pools.items():
            torch.cuda.synchronize(); t0 = time.perf_counter(); pool.stage(paths, r); torch.cuda.synchronize()
            st[k].append((time.perf_counter() - t0) * 1e3)
            t0 = time.perf_counter(); infer_files(pipe, paths, pool=pool); torch.cuda.synchronize()
            inf[k].append((time.perf_counter() - t0) * 1e3)
    n = len(paths)
    for k in pools:
        say(f"  {k:>18}: DecodePool.stage(r=128) {median(st[k]):8.1f} ms ({n / median(st[k]) * 1e3:7,.0f} files/s);  "
            f"infer_files {median(inf[k]):8.1f} ms ({n / median(inf[k]) * 1e3:7,.0f} graphs/s)")
    say(f"  (stats of the device pool: {pools['device_png'].stats}; pixels and logits identical across the three)")
    for pool in pools.values():
        pool.close()


def cap_file():
    rng = np.random.default_rng(3)
    return photo(rng, 999, 699), 999 * (1 + 3 * 699)      # raw data just under the 2 MiB cap


def stream_rate(rounds=7):
    from graphnet_classifier_b200.utils.png import decode_batch
    d, raw = cap_file()
    out = decode_batch([d])
    assert np.array_equal(out[0].cpu().numpy(), pillow(d))
    ks = []
    for _ in range(rounds):
        ops.PROFILE = ops.KernelProfile()
        decode_batch([d]); torch.cuda.synchronize()
        p = ops.PROFILE.summary()["png_decode"]
        ops.PROFILE = None
        ks.append(p["ms"] / p["calls"])
    k = median(ks)
    say(f"one file alone, 699 x 999 RGB, {len(d) / 1e6:.2f} MB compressed, {raw / 1e6:.2f} MB raw: kernels {k:.2f} ms "
        f"-> {raw / k / 1e3:.1f} MB/s of raw output per stream")


def kernel_split(name, datas, rounds=3):
    from torch.profiler import ProfilerActivity, profile
    from graphnet_classifier_b200.utils.png import decode_batch
    decode_batch(datas)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(rounds):
            decode_batch(datas)
        torch.cuda.synchronize()
    ms = {}
    for e in prof.key_averages():
        for k in ("png_inflate_kernel", "png_unfilter_kernel"):
            if k in e.key:
                total = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                ms[k] = total / e.count / 1e3
    say(f"{name}, torch.profiler: png_inflate_kernel {ms['png_inflate_kernel']:.2f} ms, "
        f"png_unfilter_kernel {ms['png_unfilter_kernel']:.2f} ms per call")


def main():
    args = sys.argv[1:]
    out_path = None
    if "--out" in args:
        i = args.index("--out"); out_path = args[i + 1]; del args[i:i + 2]
    B = int(args[0]) if args else 512
    build.build()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    say(f"GPU: {q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()}  (name, power limit, max SM clock); "
        f"host: {os.cpu_count()} cores")
    rng = np.random.default_rng(0)
    same = [photo(rng, 375, 500) for _ in range(B)]
    mixed = [photo(rng, int(h), int(w)) for h, w in rng.integers(64, 800, (B, 2))]    # all under the raw-size cap
    decode_bench("375 x 500", same)
    decode_bench("mixed sizes 64..800", mixed)
    with tempfile.TemporaryDirectory() as tmp:
        for tag, datas in (("375 x 500", same), ("mixed sizes", mixed)):
            say(f"{tag}, {B} files on disk, chunk 256:")
            pool_bench(write_files(tmp, datas, tag[:3]))
    stream_rate()
    kernel_split(f"375 x 500, {B} files", same)
    kernel_split("one file near the cap", [cap_file()[0]])
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
