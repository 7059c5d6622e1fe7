"""PNG decoded on the device (csrc/png.cu gnc_png_decode_rgb_u8 through utils/png.py) against Pillow, bit for bit: the
in-scope matrix in one batch, left-out and damaged files side by side with valid ones, hundreds of photo-like files in a
fixed number of launches, and the opt-in through DecodePool and infer_files."""
import io
import struct
import zlib

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import png as opng
from test_inflate import BitWriter, _dynamic, _lens
from test_png import _left_out, _pillow

pytestmark = pytest.mark.gpu


def _photo(rng, h, w):
    yy, xx = np.mgrid[0:h, 0:w]
    base = np.stack([(xx * 255 // w + yy // 2) % 256, (yy * 255 // h) % 256, ((xx + yy) // 3) % 256], -1)
    px = np.clip(base + rng.integers(-8, 9, (h, w, 3)), 0, 255).astype(np.uint8)
    buf = io.BytesIO()
    Image.fromarray(px).save(buf, format="PNG")
    return buf.getvalue()


def _damaged():
    """Files Pillow raises on or that the device must not claim, by name -> (bytes, Pillow accepts)."""
    rng = np.random.default_rng(5)
    px = rng.integers(0, 256, (12, 10, 3)).astype(np.uint8)
    raw = opng.filter_rows(px.reshape(12, -1), list(rng.integers(0, 5, 12)), 3)
    z = zlib.compress(raw, 9)
    far = bytearray(zlib.compress((b"\x00" + bytes(range(256)) + bytes(43)) * 12, 9))   # 12 rows of 299 grey, filter 0
    far[0], far[1] = 0x08, (31 - ((0x08 << 8) % 31)) % 31     # CINFO 0: a 256-byte window; the rows repeat 300 back
    stored = bytearray(zlib.compress(raw, 0))
    stored[5] ^= 0xff
    good = opng.write(px, 8, 2, raw_override=raw)
    i = good.index(b"IDAT")
    n = struct.unpack(">I", good[i - 4:i])[0]
    bad_idat_crc = bytearray(good)
    bad_idat_crc[i + 4 + n] ^= 1
    return {
        "bad_adler": (opng.write(px, 8, 2, zdata_override=z[:-1] + bytes([z[-1] ^ 1])), False),
        "bad_filter": (opng.write(px, 8, 2, raw_override=b"\x05" + raw[1:]), False),
        "truncated": (opng.write(px, 8, 2, zdata_override=z[:len(z) // 2]), False),
        "short_rows": (opng.write(px, 8, 2, zdata_override=zlib.compress(raw[:-31])), True),   # Pillow accepts it
        "extra_data": (opng.write(px, 8, 2, raw_override=raw + bytes(40)), True),
        # zlib (so Pillow) takes distances past the header's window; the device does not
        "window_too_small": (opng.write(np.zeros((12, 299, 1), np.uint8), 8, 0, zdata_override=bytes(far)), True),
        "block_type_3": (opng.write(px, 8, 2, zdata_override=bytes([0x78, 0x9c, 0x07, 0, 0, 0, 0, 0])), False),
        "stored_nlen": (opng.write(px, 8, 2, zdata_override=bytes(stored)), False),
        "bad_idat_crc_kept": (bytes(bad_idat_crc), True),
        "incomplete_code_set": (opng.write(px, 8, 2, zdata_override=_dynamic(_lens(257, s0=2, s65=2, s256=2), [1, 1]).zlib()), False),
        "literal_286": (opng.write(px, 8, 2, zdata_override=BitWriter().field(1, 1).field(1, 2).code(0xc6, 8).zlib()), False),
        "distance_before_output": (opng.write(px, 8, 2, zdata_override=BitWriter().field(1, 1).field(1, 2).code(0x91, 8)
                                              .code(1, 7).code(1, 5).zlib()), False),
    }


def test_matrix_in_one_batch_equals_pillow(libgnc):
    from graphnet_classifier_b200.utils.png import decode_batch
    cases = opng.matrix()
    out = decode_batch([d for _, d in cases])
    for (name, data), t in zip(cases, out):
        assert t is not None, name
        assert np.array_equal(t.cpu().numpy(), _pillow(data)), name


def test_left_out_and_damaged_files_beside_valid_ones(libgnc):
    from graphnet_classifier_b200.utils.png import decode_batch
    rng = np.random.default_rng(6)
    valid = [_photo(rng, int(h), int(w)) for h, w in rng.integers(1, 90, (10, 2))]
    damaged = _damaged()
    others = list(_left_out().values()) + [d for d, _ in damaged.values()]
    datas, expect = [], []
    for k in range(max(len(valid), len(others))):      # interleaved
        if k < len(valid):
            datas.append(valid[k]); expect.append(True)
        if k < len(others):
            datas.append(others[k]); expect.append(False)
    expect[datas.index(damaged["bad_idat_crc_kept"][0])] = True        # Pillow ignores IDAT CRCs, so does the device
    out = decode_batch(datas)
    for data, keep, t in zip(datas, expect, out):
        assert (t is not None) == keep
        if keep:
            assert np.array_equal(t.cpu().numpy(), _pillow(data))
    for name, (data, accepts) in damaged.items():
        if accepts:
            _pillow(data)
        else:
            with pytest.raises(Exception):
                _pillow(data)


def test_256_photos_in_fixed_launches(libgnc):
    from graphnet_classifier_b200 import _lib
    from graphnet_classifier_b200.utils.png import decode_batch
    rng = np.random.default_rng(7)
    datas = [_photo(rng, 375, 500) for _ in range(256)]
    counts = []
    for batch in (datas[:3], datas):
        _lib.reset_launch_count()
        out = decode_batch(batch)
        counts.append(_lib.launch_count())
    assert counts[0] == counts[1] == 2
    for data, t in zip(datas, out):
        assert np.array_equal(t.cpu().numpy(), _pillow(data))


def _mixed_files(tmp_path):
    rng = np.random.default_rng(8)
    px = [np.asarray(Image.open(io.BytesIO(_photo(rng, int(h), int(w))))) for h, w in rng.integers(20, 80, (6, 2))]
    files = []
    for k, a in enumerate(px):
        buf = io.BytesIO()
        if k % 3 == 0:
            Image.fromarray(a).save(buf, format="JPEG", quality=90)
        elif k % 3 == 1:
            Image.fromarray(a).save(buf, format="JPEG", quality=90, progressive=True)
        else:
            Image.fromarray(a).convert("CMYK").save(buf, format="JPEG", quality=90)
        files.append(buf.getvalue())
    pngs = [_photo(rng, int(h), int(w)) for h, w in rng.integers(1, 80, (7, 2))]
    pngs.append(opng.write(rng.integers(0, 4, (9, 11, 1)), 2, 3, palette=bytes(range(9)), filters=[4] * 9))
    pngs.append(_left_out()["iccp"])                                 # left out by the packer; Pillow decodes it
    pngs.append(_damaged()["extra_data"][0])                            # Pillow decodes it; the device leaves it
    paths = []
    for k, d in enumerate(files + pngs):
        p = tmp_path / f"f{k}.{'png' if d[:4] == b'\x89PNG' else 'jpg'}"
        p.write_bytes(d)
        paths.append(str(p))
    return paths, len(pngs) - 2


@pytest.mark.parametrize("device_jpeg", ["auto", False, "progressive"])
def test_decode_pool_device_png(libgnc, tmp_path, device_jpeg):
    from graphnet_classifier_b200.utils.staging import DecodePool
    paths, n_device_png = _mixed_files(tmp_path)
    r = 24
    with DecodePool(workers=2, device_jpeg=False) as pool:
        want = pool.stage(paths, r).cpu().numpy()
        want_batches = torch.cat(list(pool.batches(paths * 2, r, chunk=5))).cpu().numpy()
    with DecodePool(workers=2, device_jpeg=device_jpeg, device_png=True) as pool:
        assert np.array_equal(pool.stage(paths, r).cpu().numpy(), want)
        n_jpeg = {"auto": 2, False: 0, "progressive": 4}[device_jpeg]
        assert pool.stats == {"device_jpeg": n_jpeg, "device_png": n_device_png,
                              "host_decoded": len(paths) - n_jpeg - n_device_png}
        got = torch.cat(list(pool.batches(paths * 2, r, chunk=5)))
        assert np.array_equal(got.cpu().numpy(), want_batches)
        # without device JPEG, the files the device does not take are decoded on the worker processes, as before
        assert (pool._procs is not None) == (device_jpeg is False)


def test_corrupt_png_raises_the_same_exception(libgnc, tmp_path):
    from graphnet_classifier_b200.utils.staging import DecodePool
    paths, _ = _mixed_files(tmp_path)
    bad = tmp_path / "bad.png"
    bad.write_bytes(_damaged()["bad_adler"][0])
    types = []
    for kw in (dict(device_jpeg=False), dict(device_png=True), dict(device_jpeg=False, device_png=True)):
        with DecodePool(workers=2, **kw) as pool:
            with pytest.raises(Exception) as e:
                pool.stage(paths[:3] + [str(bad)], 16)
            types.append(type(e.value))
    assert types[0] is types[1] is types[2]


@pytest.mark.parametrize("method", ["pixel", "superpixel"])
def test_infer_files_device_png_equals_host_decode(libgnc, tmp_path, method):
    from graphnet_classifier_b200.models.GNN import CombinedModel, GraphNet
    from graphnet_classifier_b200.pipeline import GraphClassifierPipeline
    from graphnet_classifier_b200.utils.staging import DecodePool, infer_files
    paths, _ = _mixed_files(tmp_path)
    r = 16
    torch.manual_seed(0)
    if method == "pixel":
        model = CombinedModel(GraphNet(num_local_features=3, space_dim=2, out_channels=1, n_blocks=1), num_nodes=r * r)
        pipe = GraphClassifierPipeline(model.cuda().eval(), resize_value=r)
    else:
        from test_gpu_superpixel_pipeline import _models
        _, model = _models(num_nodes=20)
        pipe = GraphClassifierPipeline(model.eval(), r, method="superpixel", n_segments=20)
    with DecodePool(workers=2, device_png=True) as pool:
        dev = infer_files(pipe, paths * 2, pool=pool, chunk=6)
        assert pool.stats["device_png"] > 0
    with DecodePool(workers=2, device_jpeg=False) as pool:
        host = infer_files(pipe, paths * 2, pool=pool, chunk=6)
    assert torch.equal(dev, host)
