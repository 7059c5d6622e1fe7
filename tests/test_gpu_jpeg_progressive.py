"""Progressive JPEG decoded on the device (csrc/jpeg.cu gnc_jpeg_decode_progressive_rgb_u8 through utils/jpeg.py) against
Pillow, bit for bit: layouts and sizes side by side in one batch, restart intervals, a file without its DC refinement,
hundreds of files in one launch, mixed batches with the files left to the host, and the opt-in through DecodePool and
infer_files."""

import numpy as np
import pytest
import torch
from PIL import Image

from oracle.jpeg_progressive import decode_progressive
from test_jpeg_progressive import _jpeg, left_out_files, pillow, without_scan

pytestmark = pytest.mark.gpu

CASES = [(32, 32, dict(quality=90)), (33, 47, dict(quality=75)), (17, 23, dict(quality=95, subsampling=0)),
         (40, 50, dict(quality=60, subsampling=1)), (31, 65, dict(quality=90, gray=True)),
         (50, 70, dict(quality=80, restart_marker_blocks=3)), (57, 91, dict(quality=80, restart_marker_rows=1, subsampling=1)),
         (45, 61, dict(quality=85, restart_marker_blocks=1, gray=True)), (20, 3, dict(quality=90)), (5, 4, dict(quality=90)),
         (1, 1, dict(quality=90)), (8, 8, dict(quality=50, subsampling=0)), (100, 150, dict(quality=5)),
         (16, 16, dict(quality=100, subsampling=2)), (375, 500, dict(quality=90)), (600, 800, dict(quality=25)),
         (97, 1201, dict(quality=90, subsampling=2)), (512, 512, dict(quality=99, noise=90)),
         (400, 300, dict(quality=92, gray=True)), (333, 517, dict(quality=70, subsampling=1, restart_marker_rows=2))]


def _cases():
    rng = np.random.default_rng(11)
    datas = [_jpeg(rng, h, w, **dict(kw)) for h, w, kw in CASES]
    datas.append(without_scan(_jpeg(rng, 61, 77, quality=90), 6))         # no DC refinement: kept, half-precision DC
    return datas


@pytest.mark.parametrize("per_warp", [32, 4])
def test_one_batch_equals_pillow(libgnc, per_warp):
    from graphnet_classifier_b200.utils.jpeg import decode_batch
    datas = _cases()
    libgnc.gnc_debug_jpeg_chains_per_warp(per_warp)
    try:
        out = decode_batch(datas, progressive=True)
        torch.cuda.synchronize()
    finally:
        libgnc.gnc_debug_jpeg_chains_per_warp(0)
    for i, (data, t) in enumerate(zip(datas, out)):
        ref = pillow(data)
        assert t is not None, i
        got = t.cpu().numpy()
        assert got.shape == ref.shape and np.array_equal(got, ref), (i, int(np.abs(got.astype(int) - ref).max()))
        if ref.shape[0] * ref.shape[1] <= 6000:
            assert np.array_equal(decode_progressive(data), ref), i


def test_many_files_share_a_launch(libgnc):
    from graphnet_classifier_b200.utils.jpeg import decode_batch
    rng = np.random.default_rng(12)
    datas = [_jpeg(rng, 375, 500, quality=int(q)) for q in rng.integers(60, 100, 256)]
    out = decode_batch(datas, progressive=True)
    for i, (data, t) in enumerate(zip(datas, out)):
        assert t is not None and np.array_equal(t.cpu().numpy(), pillow(data)), i


def _mixed():
    rng = np.random.default_rng(13)
    files = left_out_files()
    datas = [_jpeg(rng, 40, 56, quality=90, progressive=False), _jpeg(rng, 40, 56, quality=90),
             files["png"], files["cmyk"], files["cut_after_3"], _jpeg(rng, 120, 90, quality=70, subsampling=0),
             _jpeg(rng, 33, 47, quality=80, progressive=False, subsampling=1), _jpeg(rng, 50, 50, quality=95, gray=True)]
    device = [True, True, False, False, False, True, True, True]
    progressive = [False, True, False, False, False, True, False, True]
    return datas, device, progressive


def test_mixed_batch(libgnc):
    from graphnet_classifier_b200.utils.jpeg import decode_batch
    datas, device, progressive = _mixed()
    staging = {}
    first = decode_batch(datas, staging=staging, progressive=True)
    second = decode_batch(datas, staging=staging, progressive=True)
    for data, dev, a, b in zip(datas, device, first, second):
        if not dev:
            assert a is None and b is None
            continue
        assert np.array_equal(a.cpu().numpy(), pillow(data)) and torch.equal(a, b)
    default = decode_batch(datas)
    for prog, dev, t in zip(progressive, device, default):
        assert (t is not None) == (dev and not prog)


def _write(tmp_path, datas):
    paths = []
    for i, d in enumerate(datas):
        p = tmp_path / f"f{i}.img"
        p.write_bytes(d)
        paths.append(str(p))
    return paths


def test_decode_pool_progressive(libgnc, tmp_path):
    from graphnet_classifier_b200.utils.staging import DecodePool
    datas, device, _ = _mixed()
    paths = _write(tmp_path, datas)
    r = 24
    want = np.stack([np.array(Image.open(p).convert("RGB").resize((r, r))) for p in paths])
    with DecodePool(workers=2, device_jpeg="progressive") as pool:
        assert np.array_equal(pool.stage(paths, r).cpu().numpy(), want)
        assert pool.stats == {"device_jpeg": sum(device), "host_decoded": len(paths) - sum(device)}
        got = torch.cat(list(pool.batches(paths * 3, r, chunk=5)))
        assert np.array_equal(got.cpu().numpy(), np.concatenate([want] * 3))


def test_infer_files_progressive_equals_host_decode(libgnc, tmp_path):
    from graphnet_classifier_b200.models.GNN import CombinedModel, GraphNet
    from graphnet_classifier_b200.pipeline import GraphClassifierPipeline
    from graphnet_classifier_b200.utils.staging import DecodePool, infer_files
    datas, _, _ = _mixed()
    paths = _write(tmp_path, datas) * 2
    torch.manual_seed(0)
    r = 16
    model = CombinedModel(GraphNet(num_local_features=3, space_dim=2, out_channels=1, n_blocks=1), num_nodes=r * r).cuda().eval()
    pipe = GraphClassifierPipeline(model, resize_value=r)
    with DecodePool(workers=2, device_jpeg="progressive") as pool:
        dev = infer_files(pipe, paths, pool=pool, chunk=6)
        assert pool.stats["device_jpeg"] > 0
    with DecodePool(workers=2, device_jpeg=False) as pool:
        host = infer_files(pipe, paths, pool=pool, chunk=6)
    assert torch.equal(dev, host)
