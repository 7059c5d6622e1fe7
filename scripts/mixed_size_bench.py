#!/usr/bin/env python
"""Mixed-size photo collections through the device resize and the files -> logits path.

    mixed_size_bench.py [N] [--rounds R]

N seeded JPEG files (quality 90) with H, W drawn uniformly from [160, 900], and N files of 375 x 500 for comparison.
Two measurements, each alternating the two staging forms in the same process and reporting medians:
  * resize alone, on one device-decoded batch: the per-shape form (one ``ops.resize_bicubic`` per shape group, a
    ``torch.stack`` and a scatter into the output, as DecodePool staged a chunk before the ragged resize) against one
    ``ops.resize_bicubic_ragged`` call; CUDA-event time, host wall time and kernel launches (libgnc's launch counter);
  * end to end, ``infer_files`` at resize 128 and chunk 256 with device JPEG decode, the per-shape staging put back by
    a local switch (``DecodePool._upload_jpeg`` replaced for the duration of the call).
Outputs of the two forms are compared bit for bit.  The GPU's name and power limit are printed first."""
import argparse, io, os, shutil, subprocess, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from PIL import Image
from graphnet_classifier_b200 import _lib, build, ops
from graphnet_classifier_b200.utils import jpeg as gjpeg
from graphnet_classifier_b200.utils import staging


def make_files(n, mixed, seed):
    rng = np.random.default_rng(seed)
    datas = []
    for _ in range(n):
        h, w = (int(v) for v in rng.integers(160, 901, 2)) if mixed else (375, 500)
        low = rng.integers(0, 256, (h // 16 + 2, w // 16 + 2, 3), dtype=np.uint8)
        buf = io.BytesIO()
        Image.fromarray(low).resize((w, h), Image.BICUBIC).save(buf, format="JPEG", quality=90)
        datas.append(buf.getvalue())
    return datas


def per_shape_resize(imgs, r, device):
    """The staging of a chunk before the ragged resize: one group per shape, stacked, resized, scattered."""
    groups = {}
    for i, t in enumerate(imgs):
        groups.setdefault(tuple(t.shape), []).append(i)
    n = len(imgs)
    out = None
    for shape, idxs in groups.items():
        if len(idxs) == n and all(imgs[i].data_ptr() + imgs[i].numel() == imgs[i + 1].data_ptr() for i in range(n - 1)):
            batch = torch.as_strided(imgs[0], (n, *shape), (imgs[0].numel(), shape[1] * 3, 3, 1))
        else:
            batch = torch.stack([imgs[i] for i in idxs])
        px = batch if (shape[0] == r and shape[1] == r) else ops.resize_bicubic(batch, r, r)
        if len(groups) == 1:
            return px
        if out is None:
            out = torch.empty(n, r, r, 3, dtype=torch.uint8, device=device)
        out[torch.as_tensor(idxs, device=device)] = px
    return out


def per_shape_upload_jpeg(self, chunk, resize_value):
    """DecodePool._upload_jpeg with the per-shape resize above."""
    pairs, host = chunk["jpeg"], chunk["host"]
    datas = [d if i not in host else b"" for i, (d, _) in enumerate(pairs)]
    imgs = gjpeg.decode_batch(datas, self.device, staging=self._jpeg_staging[chunk["slot"]], progressive=self.progressive_jpeg)
    late = [i for i, t in enumerate(imgs) if t is None and i not in host]
    if late:
        host = dict(host)
        host.update(zip(late, self.pool.map(staging._decode, [chunk["paths"][i] for i in late])))
    self.stats["device_jpeg"] += len(imgs) - len(host)
    self.stats["host_decoded"] += len(host)
    for i, a in host.items():
        imgs[i] = torch.from_numpy(np.array(a, dtype=np.uint8)).to(self.device)
    return per_shape_resize(imgs, int(resize_value), self.device)


def med(xs):
    return sorted(xs)[len(xs) // 2]


def resize_alone(name, datas, r, rounds):
    dev = torch.device("cuda")
    imgs = gjpeg.decode_batch(datas, dev)
    forms = {"per-shape": lambda: per_shape_resize(imgs, r, dev), "ragged": lambda: ops.resize_bicubic_ragged(imgs, r, r)}
    outs = {k: f() for k, f in forms.items()}
    same = torch.equal(outs["per-shape"], outs["ragged"])
    times = {k: ([], [], []) for k in forms}
    for _ in range(rounds):
        for k, f in forms.items():
            torch.cuda.synchronize()
            n0 = _lib.launch_count()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            s.record(); f(); e.record()
            torch.cuda.synchronize()
            times[k][0].append(s.elapsed_time(e))
            times[k][1].append((time.perf_counter() - t0) * 1e3)
            times[k][2].append(_lib.launch_count() - n0)
    shapes = len({tuple(t.shape) for t in imgs})
    print(f"resize alone, {name}: {len(imgs)} device-decoded images, {shapes} shapes -> {r} x {r}; outputs equal: {same}")
    for k in forms:
        ev, wall, launches = times[k]
        print(f"  {k:9s}: {med(ev):8.3f} ms CUDA events (range {min(ev):.3f} .. {max(ev):.3f}), {med(wall):8.3f} ms host wall, "
              f"{med(launches)} kernel launches")
    return same


def end_to_end(name, paths, pipe, pool, rounds, chunk=256):
    forms = {"per-shape": per_shape_upload_jpeg, "ragged": staging.DecodePool._upload_jpeg}
    logits, times = {}, {k: [] for k in forms}
    for rnd in range(rounds + 1):                         # round 0 warms buffers, resize tables and topology caches
        for k, upload in forms.items():
            pool._upload_jpeg = upload.__get__(pool)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = staging.infer_files(pipe, paths, pool=pool, chunk=chunk).cpu()
            dt = (time.perf_counter() - t0) * 1e3
            if rnd:
                times[k].append(dt)
            logits[k] = out
    del pool._upload_jpeg
    same = torch.equal(logits["per-shape"], logits["ragged"])
    print(f"infer_files, {name}: {len(paths)} files, resize {pipe.resize_value}, chunk {chunk}; logits equal: {same}")
    for k, ts in times.items():
        m = med(ts)
        print(f"  {k:9s}: {m:8.2f} ms -> {len(paths) / m * 1e3:,.0f} graphs/s (range {min(ts):.2f} .. {max(ts):.2f})")
    return same


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("n", type=int, nargs="?", default=512)
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("mixed_size_bench.py measures on a CUDA device; none found")
    build.build()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"GPU: {q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()}  (name, power limit, max SM clock)")
    from graphnet_classifier_b200.models.GNN import CombinedModel, GraphNet
    from graphnet_classifier_b200.pipeline import GraphClassifierPipeline
    r = 128
    torch.manual_seed(0)
    model = CombinedModel(GraphNet(num_local_features=3, space_dim=2, out_channels=1, n_blocks=3), num_nodes=r * r).cuda().eval()
    pipe = GraphClassifierPipeline(model, resize_value=r)
    sets = {"mixed H, W in [160, 900]": make_files(args.n, True, 1), "uniform 375 x 500": make_files(args.n, False, 2)}
    ok = True
    for name, datas in sets.items():
        ok &= resize_alone(name, datas[:256], r, args.rounds)
    d = tempfile.mkdtemp()
    try:
        with staging.DecodePool() as pool:
            for j, (name, datas) in enumerate(sets.items()):
                paths = []
                for i, data in enumerate(datas):
                    p = os.path.join(d, f"{j}_{i}.jpg")
                    with open(p, "wb") as f:
                        f.write(data)
                    paths.append(p)
                ok &= end_to_end(name, paths, pipe, pool, args.rounds)
    finally:
        shutil.rmtree(d, ignore_errors=True)
    if not ok:
        sys.exit("the two staging forms differ")


if __name__ == "__main__":
    main()
