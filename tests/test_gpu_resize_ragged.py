"""GPU: ragged batches through the Pillow-exact resize (csrc/resize.cu gnc_resize_bicubic_ragged_u8, ops.resize_bicubic_ragged):
the device coefficient tables against the host's int for int, images of many sizes against Pillow and the one-shape
resize bit for bit, DecodePool and GraphClassifierPipeline on mixed sizes, and a launch count that does not grow with the
number of shapes."""
import io

import numpy as np
import pytest
import torch
from PIL import Image

from test_gpu_superpixel_pipeline import _models, _smooth_images
from test_jpeg_progressive import _jpeg

pytestmark = pytest.mark.gpu

IN_SIZES = list(range(1, 1101)) + [2999, 3000, 4000, 12000]
OUT_SIZES = [1, 2, 3, 24, 64, 100, 127, 128, 129, 256, 333, 512]


def _pillow(a, oh, ow):
    return np.asarray(Image.fromarray(a).resize((ow, oh)))


def _device_tables(libgnc, shapes, oh, ow):
    """Runs the C entry point on images of `shapes` (zeros) and returns (records, tables) from the device."""
    from graphnet_classifier_b200 import ops
    rec, n_tables, h_rows, max_w = ops._ragged_plan([s[0] for s in shapes], [s[1] for s in shapes], oh, ow)
    offs = np.concatenate([[0], np.cumsum([3 * h * w for h, w in shapes])])
    buf = torch.zeros(int(offs[-1]), dtype=torch.uint8, device="cuda")
    rec["src"] = buf.data_ptr() + offs[:-1]
    rec["pitch"] = [3 * w for _, w in shapes]
    recs = torch.from_numpy(rec.view(np.uint8).copy()).cuda()
    tables = torch.full((max(n_tables, 1),), -7, dtype=torch.int32, device="cuda")
    tmp = torch.empty(max(h_rows * 3 * ow, 1), dtype=torch.uint8, device="cuda")
    dst = torch.empty(len(shapes), oh, ow, 3, dtype=torch.uint8, device="cuda")
    assert libgnc.gnc_resize_bicubic_ragged_u8(recs.data_ptr(), len(shapes), oh, ow, h_rows, max_w, tables.data_ptr(),
                                               tmp.data_ptr(), dst.data_ptr(), torch.cuda.current_stream().cuda_stream) == 0
    assert bool((dst == 0).all())
    return rec, tables.cpu().numpy()


@pytest.mark.parametrize("out", OUT_SIZES)
def test_device_tables_equal_host_coeffs(libgnc, out):
    """Both axes, every in size against `out`: bounds and kk equal gnc_resize_bicubic_coeffs int for int; an axis whose
    size is already `out` has no table (Pillow does not filter it)."""
    for axis in ("y", "x"):
        shapes = [(n, 1) for n in IN_SIZES] if axis == "y" else [(1, n) for n in IN_SIZES]
        oh, ow = (out, 1) if axis == "y" else (1, out)
        rec, tables = _device_tables(libgnc, shapes, oh, ow)
        for i, n in enumerate(IN_SIZES):
            ks, tab = int(rec["ksize_" + axis][i]), int(rec["tab_" + axis][i])
            if n == out:
                assert ks == 0, n
                continue
            assert ks == libgnc.gnc_resize_bicubic_ksize(n, out), n
            bounds = np.empty((out, 2), np.int32)
            kk = np.empty((out, ks), np.int32)
            assert libgnc.gnc_resize_bicubic_coeffs(n, out, bounds.ctypes.data, kk.ctypes.data) == 0
            got_b = tables[tab:tab + 2 * out].reshape(out, 2)
            got_k = tables[tab + 2 * out:tab + out * (2 + ks)].reshape(out, ks)
            assert np.array_equal(got_b, bounds), (axis, n, out)
            assert np.array_equal(got_k, kk), (axis, n, out)


def _check(images_np, views, oh, ow):
    from graphnet_classifier_b200 import ops
    got = ops.resize_bicubic_ragged(views, oh, ow)
    assert got.shape == (len(views), oh, ow, 3) and got.dtype == torch.uint8
    got = got.cpu().numpy()
    for i, (a, v) in enumerate(zip(images_np, views)):
        assert np.array_equal(got[i], _pillow(a, oh, ow)), (i, a.shape, oh, ow)
        assert np.array_equal(got[i], ops.resize_bicubic(v, oh, ow).cpu().numpy()), (i, a.shape)


@pytest.mark.parametrize("oh,ow", [(128, 128), (48, 80), (97, 31)])
def test_ragged_batch_equals_pillow(libgnc, oh, ow):
    rng = np.random.default_rng(oh * 1000 + ow)
    shapes = [(1, 1), (1, 97), (97, 1), (oh, ow), (oh, 50), (60, ow), (375, 500), (500, 375), (33, 35), (2, 3),
              (oh + 1, ow - 1), (900, 160), (4, 4000)]
    imgs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in shapes]
    imgs[6][:100] = 255                                       # saturated regions: overshoot is clamped
    imgs[6][100:200] = 0
    _check(imgs, [torch.from_numpy(a).cuda() for a in imgs], oh, ow)


def test_large_photo_among_small_ones(libgnc):
    rng = np.random.default_rng(5)
    imgs = [rng.integers(0, 256, (3000, 4000, 3), dtype=np.uint8), rng.integers(0, 256, (37, 41, 3), dtype=np.uint8),
            rng.integers(0, 256, (128, 128, 3), dtype=np.uint8)]
    _check(imgs, [torch.from_numpy(a).cuda() for a in imgs], 128, 128)


def test_views_at_odd_offsets_in_one_buffer(libgnc):
    """The JPEG decoder's layout: images back to back in one packed RGB buffer at 3 * pixel_offset, here starting at an
    odd byte; plus crops of a larger image (row pitch not a multiple of 4) and a non-contiguous view."""
    rng = np.random.default_rng(8)
    shapes = [(45, 61), (3, 7), (130, 129), (1, 5), (77, 200)]
    imgs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in shapes]
    flat = torch.zeros(1 + sum(a.size for a in imgs), dtype=torch.uint8, device="cuda")
    views, off = [], 1
    for a in imgs:
        flat[off:off + a.size] = torch.from_numpy(a.reshape(-1)).cuda()
        views.append(flat[off:off + a.size].view(*a.shape))
        off += a.size
    big = rng.integers(0, 256, (90, 110, 3), dtype=np.uint8)
    dbig = torch.from_numpy(big).cuda()
    imgs += [np.ascontiguousarray(big[3:64, 5:82]), np.ascontiguousarray(big[::2, 1::3])]
    views += [dbig[3:64, 5:82], dbig[::2, 1::3]]
    _check(imgs, views, 64, 48)


def test_one_and_no_images(libgnc):
    from graphnet_classifier_b200 import ops
    a = np.random.default_rng(1).integers(0, 256, (51, 77, 3), dtype=np.uint8)
    _check([a], [torch.from_numpy(a).cuda()], 20, 30)
    empty = ops.resize_bicubic_ragged([], 20, 30)
    assert empty.shape == (0, 20, 30, 3) and empty.is_cuda
    with pytest.raises(ValueError):
        ops.resize_bicubic_ragged([torch.zeros(4, 4, 4, dtype=torch.uint8, device="cuda")], 8)


def test_launches_do_not_grow_with_shapes(libgnc):
    from graphnet_classifier_b200 import _lib, ops
    rng = np.random.default_rng(2)
    counts = []
    for n_shapes in (2, 64):
        views = [torch.from_numpy(rng.integers(0, 256, (100 + i, 300 - 2 * i, 3), dtype=np.uint8)).cuda()
                 for i in range(n_shapes)]
        torch.cuda.synchronize()
        before = _lib.launch_count()
        ops.resize_bicubic_ragged(views, 128, 128)
        counts.append(_lib.launch_count() - before)
    assert counts[0] == counts[1] <= 3, counts


def _folder(tmp_path):
    """Mixed-size baseline and progressive JPEG files, PNG and CMYK JPEG files."""
    rng = np.random.default_rng(31)
    datas, kinds = [], []
    for k in range(12):
        h, w = (int(v) for v in rng.integers(20, 160, 2))
        datas.append(_jpeg(rng, h, w, quality=int(rng.integers(60, 96)), progressive=bool(k % 3 == 1)))
        kinds.append("progressive" if k % 3 == 1 else "baseline")
    datas.append(_jpeg(rng, 24, 24, quality=90, progressive=False))         # already the target size
    kinds.append("baseline")
    for fmt, mode in (("PNG", "RGB"), ("JPEG", "CMYK")):
        arr = rng.integers(0, 256, (int(rng.integers(20, 90)), int(rng.integers(20, 90)), 3), dtype=np.uint8)
        buf = io.BytesIO()
        Image.fromarray(arr).convert(mode).save(buf, format=fmt)
        datas.append(buf.getvalue())
        kinds.append(fmt.lower())
    paths = []
    for i, d in enumerate(datas):
        p = tmp_path / f"f{i}.img"
        p.write_bytes(d)
        paths.append(str(p))
    return paths, kinds


@pytest.mark.parametrize("device_jpeg,processes", [(True, True), ("progressive", True), (False, True), (False, False)])
def test_decode_pool_mixed_sizes(libgnc, tmp_path, device_jpeg, processes):
    from graphnet_classifier_b200.utils.staging import DecodePool
    paths, kinds = _folder(tmp_path)
    r = 24
    want = np.stack([np.array(Image.open(p).convert("RGB").resize((r, r))) for p in paths])
    on_device = {True: ("baseline",), "progressive": ("baseline", "progressive"), False: ()}[device_jpeg]
    with DecodePool(workers=2, device_jpeg=device_jpeg, processes=processes) as pool:
        assert np.array_equal(pool.stage(paths, r).cpu().numpy(), want)
        n_dev = sum(k in on_device for k in kinds) if device_jpeg else 0
        n_host = len(paths) - n_dev if device_jpeg else 0
        assert pool.stats == {"device_jpeg": n_dev, "host_decoded": n_host}
        got = torch.cat(list(pool.batches(paths * 2, r, chunk=7)))
        assert np.array_equal(got.cpu().numpy(), np.concatenate([want] * 2))


@pytest.mark.parametrize("method", ["pixel", "superpixel"])
def test_pipeline_mixed_sizes_equal_pillow_stack(libgnc, tmp_path, method):
    from graphnet_classifier_b200.models.GNN import CombinedModel, GraphNet
    from graphnet_classifier_b200.pipeline import GraphClassifierPipeline
    from graphnet_classifier_b200.utils.staging import DecodePool, infer_files
    r = 32
    if method == "pixel":
        torch.manual_seed(0)
        model = CombinedModel(GraphNet(num_local_features=3, space_dim=2, out_channels=1, n_blocks=1), num_nodes=r * r).cuda().eval()
        pipe = GraphClassifierPipeline(model, resize_value=r)
    else:
        _, model = _models(num_nodes=20)
        pipe = GraphClassifierPipeline(model.eval(), r, method="superpixel", n_segments=20)
    rng = np.random.default_rng(4)
    raw = [_smooth_images(rng, 1, int(h), int(w), noise=20)[0] for h, w in rng.integers(10, 120, (9, 2))]
    raw.append(_smooth_images(rng, 1, r, r)[0])
    pre = torch.from_numpy(np.stack([_pillow(a, r, r) for a in raw]))
    want = pipe.infer(pre)
    assert torch.equal(pipe.infer([torch.from_numpy(a) for a in raw]), want)
    assert torch.equal(pipe.infer(raw), want)
    paths = []
    for i, a in enumerate(raw):
        p = tmp_path / f"im{i}.png"
        Image.fromarray(a).save(p)
        paths.append(str(p))
    with DecodePool(workers=2) as pool:
        got = infer_files(pipe, paths, pool=pool, chunk=4)
    assert torch.equal(got, torch.cat([pipe.infer(pre[lo:lo + 4]) for lo in range(0, len(raw), 4)]))
