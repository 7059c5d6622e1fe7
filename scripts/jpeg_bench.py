#!/usr/bin/env python
"""Device JPEG decoder (csrc/jpeg.cu) alone: B synthetic 375 x 500 quality-90 files, bytes in host memory -> RGB pixels
in HBM; checked against Pillow on the first files; CUDA events, median of 5.

    jpeg_bench.py [B] [--progressive]

--progressive: the same files saved progressive, written to a temporary directory; reports the full decode_batch call
and the kernels alone (with the chain count and each chains-per-warp mapping of the entropy kernel), and
DecodePool.stage over the paths with host decoding (worker processes) and with device_jpeg="progressive", in
interleaved rounds (medians), with the GPU's name and power limit."""
import io, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from PIL import Image
from graphnet_classifier_b200 import build, ops


def make_files(B, progressive):
    rng = np.random.default_rng(0)
    datas = []
    for i in range(B):
        low = rng.integers(0, 256, (375 // 16 + 2, 500 // 16 + 2, 3), dtype=np.uint8)
        buf = io.BytesIO()
        Image.fromarray(low).resize((500, 375), Image.BICUBIC).save(buf, format="JPEG", quality=90, progressive=progressive)
        datas.append(buf.getvalue())
    return datas


def baseline_bench(datas):
    B = len(datas)
    st = {}
    out = gjpeg.decode_batch(datas, staging=st)
    for d, t in list(zip(datas, out))[:8]:
        assert np.array_equal(t.cpu().numpy(), np.asarray(Image.open(io.BytesIO(d)).convert("RGB")))
    ts = []
    for _ in range(5):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); gjpeg.decode_batch(datas, staging=st); e.record(); torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    ms = sorted(ts)[2]
    ops.PROFILE = ops.KernelProfile()
    for _ in range(3):
        gjpeg.decode_batch(datas, staging=st)
    prof = ops.PROFILE.summary()["jpeg_decode"]
    ops.PROFILE = None
    print(f"device kernels alone (memset + entropy + IDCT + upsampling/colour): {prof['ms'] / prof['calls']:.2f} ms per call "
          f"-> {B / (prof['ms'] / prof['calls']) * 1e3:,.0f} images/s; the rest of the call is host work (descriptor table, copies into pinned memory)")
    print(f"{B} files of {sum(map(len, datas)) / B / 1e3:.1f} KB: {ms:.2f} ms -> {B / ms * 1e3:,.0f} images/s (bit-identical to Pillow on the checked files)")


def progressive_bench(datas, rounds=5, r=128):
    import subprocess, tempfile
    from graphnet_classifier_b200 import _lib
    from graphnet_classifier_b200.utils.staging import DecodePool
    lib = _lib.load()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"GPU: {q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()}  (name, power limit, max SM clock)")
    st = {}
    out = gjpeg.decode_batch(datas, staging=st, progressive=True)
    torch.cuda.synchronize()
    bad = sum(t is None or not np.array_equal(t.cpu().numpy(), np.asarray(Image.open(io.BytesIO(d)).convert("RGB")))
              for d, t in zip(datas, out))
    n_chains = 4 * len(datas)                       # Pillow's colour script: DC, Y AC, Cb AC, Cr AC
    print(f"{len(datas)} progressive files of {sum(map(len, datas)) / len(datas) / 1e3:.1f} KB, {n_chains} chains; "
          f"{bad} differ from Pillow")

    def call():
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); gjpeg.decode_batch(datas, staging=st, progressive=True); e.record(); torch.cuda.synchronize()
        return s.elapsed_time(e)

    def kernels(per_warp):
        lib.gnc_debug_jpeg_chains_per_warp(per_warp)
        ops.PROFILE = ops.KernelProfile()
        for _ in range(3):
            gjpeg.decode_batch(datas, staging=st, progressive=True)
        prof = ops.PROFILE.summary()["jpeg_decode_progressive"]
        ops.PROFILE = None
        lib.gnc_debug_jpeg_chains_per_warp(0)
        return prof["ms"] / prof["calls"]

    with tempfile.TemporaryDirectory() as tmp:
        paths = []
        for i, d in enumerate(datas):
            paths.append(os.path.join(tmp, f"{i}.jpg"))
            with open(paths[-1], "wb") as f:
                f.write(d)
        host, dev = DecodePool(device_jpeg=False), DecodePool(device_jpeg="progressive")
        pools = {"host processes": host, "device (progressive)": dev}
        try:
            want = host.stage(paths, r)
            assert torch.equal(dev.stage(paths, r), want)            # also warms both pools up
            per_warps = (32, 16, 8, 4, 2, 1)
            times = {k: [] for k in ["call"] + [f"kernels {w}" for w in per_warps] + list(pools)}
            for _ in range(rounds):                                     # interleaved rounds
                times["call"].append(call())
                for w in per_warps:
                    times[f"kernels {w}"].append(kernels(w))
                for name, pool in pools.items():
                    torch.cuda.synchronize()
                    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    s.record(); pool.stage(paths, r); e.record(); torch.cuda.synchronize()
                    times[name].append(s.elapsed_time(e))
        finally:
            host.close(); dev.close()
    med = {k: float(np.median(v)) for k, v in times.items()}
    n = len(datas)
    print(f"medians of {rounds} interleaved rounds, {n} files, {n_chains} chains:")
    print(f"  decode_batch(progressive=True), full call: {med['call']:.2f} ms -> {n / med['call'] * 1e3:,.0f} files/s")
    for w in per_warps:
        k = med[f"kernels {w}"]
        print(f"  kernels alone (memset + entropy + IDCT + colour), {w:2d} chains per warp: {k:.2f} ms -> {n / k * 1e3:,.0f} files/s")
    for name in pools:
        print(f"  DecodePool.stage({n} paths, {r}) {name}: {med[name]:.2f} ms -> {n / med[name] * 1e3:,.0f} files/s "
              f"(range {min(times[name]):.2f} .. {max(times[name]):.2f})")


if __name__ == "__main__":          # DecodePool's worker processes (spawn) import this module: nothing runs there
    build.build()
    from graphnet_classifier_b200.utils import jpeg as gjpeg
    progressive = "--progressive" in sys.argv
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    datas = make_files(int(args[0]) if args else 512, progressive)
    (progressive_bench if progressive else baseline_bench)(datas)
