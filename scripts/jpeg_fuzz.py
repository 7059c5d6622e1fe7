#!/usr/bin/env python
"""Randomised check of the device JPEG decoder against Pillow: N files of random size (1 .. 700), content (smooth, noisy,
flat, text-like edges), quality (5 .. 100), chroma layout, Huffman-table optimisation and restart interval, decoded in
batches of 64 (images of every kind side by side).  Every pixel must match.

    jpeg_fuzz.py [N] [SEED] [--progressive]

--progressive: about half the files are saved progressive (Pillow's script, also with restart intervals) and the batches
go through decode_batch(..., progressive=True); every file must come back decoded."""
import io, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from PIL import Image
from graphnet_classifier_b200 import build
build.build()
from graphnet_classifier_b200.utils import jpeg as gjpeg
PROGRESSIVE = "--progressive" in sys.argv
args = [a for a in sys.argv[1:] if not a.startswith("--")]
N = int(args[0]) if args else 256
if PROGRESSIVE:
    from PIL import ImageFile
    ImageFile.MAXBLOCK = 1 << 25        # Pillow's progressive encoder buffer is W * H bytes: noisy 4:4:4 content overflows it
rng = np.random.default_rng(int(args[1]) if len(args) > 1 else 0)


def image(h, w):
    kind = rng.integers(0, 4)
    if kind == 0:
        low = rng.integers(0, 256, (h // 16 + 2, w // 16 + 2, 3), dtype=np.uint8)
        a = np.asarray(Image.fromarray(low).resize((w, h), Image.BICUBIC)).astype(int)
    elif kind == 1:
        a = rng.integers(0, 256, (h, w, 3))
    elif kind == 2:
        a = np.full((h, w, 3), rng.integers(0, 256, 3))
    else:
        a = np.where(rng.random((h, w, 1)) < 0.1, 0, 255) * np.ones((1, 1, 3), int)
    return np.clip(a + rng.integers(-6, 7, (h, w, 3)), 0, 255).astype(np.uint8)


datas, kws = [], []
for i in range(N):
    h, w = int(rng.integers(1, 700)), int(rng.integers(1, 700))
    kw = dict(quality=int(rng.integers(5, 101)), subsampling=int(rng.integers(0, 3)), optimize=bool(rng.integers(0, 2)))
    if rng.random() < 0.15:
        kw["restart_marker_blocks"] = int(rng.integers(1, 20))
    if PROGRESSIVE and rng.random() < 0.5:
        kw["progressive"] = True
        if rng.random() < 0.1:
            kw["restart_marker_rows"] = int(rng.integers(1, 4))
    im = Image.fromarray(image(h, w))
    if rng.random() < 0.15:
        im = im.convert("L"); kw.pop("subsampling")
    buf = io.BytesIO()
    try:
        im.save(buf, format="JPEG", **kw)
    except OSError:                               # Pillow's encoder rejects a few parameter combinations
        kw.pop("restart_marker_blocks", None); kw.pop("restart_marker_rows", None); kw["optimize"] = False
        buf = io.BytesIO(); im.save(buf, format="JPEG", **kw)
    datas.append(buf.getvalue()); kws.append((h, w, kw))
bad = big = 0
for lo in range(0, N, 64):
    out = gjpeg.decode_batch(datas[lo:lo + 64], progressive=PROGRESSIVE)
    torch.cuda.synchronize()
    for d, t, kw in zip(datas[lo:lo + 64], out, kws[lo:lo + 64]):
        ref = np.asarray(Image.open(io.BytesIO(d)).convert("RGB"))
        big += len(d) >= 4096 + 700
        if t is None or t.shape != ref.shape or not np.array_equal(t.cpu().numpy(), ref):
            bad += 1
            print("MISMATCH", kw, None if t is None else int(np.abs(t.cpu().numpy().astype(int) - ref).max()))
n_prog = sum(bool(kw.get("progressive")) for _, _, kw in kws)
print(f"{N} files ({n_prog} progressive, {big} large enough for the parallel entropy decoder): {bad} mismatches")
sys.exit(1 if bad else 0)
