"""CPU: the PNG restatement (oracle/png.py) equals Pillow on the in-scope matrix, and gnc_png_pack accepts exactly the
in-scope files and leaves every left-out kind to the host."""
import ctypes
import io
import struct
import zlib

import numpy as np
import pytest
from PIL import Image

from oracle import png as opng


def _pillow(data):
    return np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))


@pytest.fixture(scope="module")
def cases():
    return opng.matrix()


def test_oracle_equals_pillow_on_the_matrix(cases):
    for name, data in cases:
        ref = _pillow(data)
        got = opng.decode(data)
        assert got is not None, name
        assert got.shape == ref.shape and np.array_equal(got, ref), name


def test_conversion_table():
    """The rows of include/gnc.h's conversion table, on hand-picked samples."""
    v16 = np.array([[0x0102, 0x01ff, 0x8000, 0xffff, 0, 1, 200, 255]], np.uint16)
    assert _pillow(opng.write(v16[:, :, None], 16, 0))[0, :, 0].tolist() == [255, 255, 255, 255, 0, 1, 200, 255]
    assert _pillow(opng.write(np.repeat(v16[:, :, None], 3, 2), 16, 2))[0, :4, 0].tolist() == [1, 1, 128, 255]
    assert _pillow(opng.write(np.repeat(v16[:, :, None], 2, 2), 16, 4))[0, :4, 0].tolist() == [1, 1, 128, 255]
    assert _pillow(opng.write(np.array([[[0], [1], [2], [3]]]), 2, 0))[0, :, 0].tolist() == [0, 85, 170, 255]
    assert _pillow(opng.write(np.array([[[0], [15], [8]]]), 4, 0))[0, :, 0].tolist() == [0, 255, 136]
    assert _pillow(opng.write(np.array([[[0], [1]]]), 1, 0))[0, :, 0].tolist() == [0, 255]
    short = _pillow(opng.write(np.array([[[0], [1], [2], [255]]], np.uint8), 8, 3, palette=bytes([10, 20, 30, 40, 50, 60])))
    assert short[0].tolist() == [[10, 20, 30], [40, 50, 60], [0, 0, 0], [0, 0, 0]]


def test_large_photo_like_image():
    rng = np.random.default_rng(1)
    yy, xx = np.mgrid[0:1500, 0:2000]
    px = np.clip(np.stack([(xx // 8 + yy // 6) % 256, (xx // 5) % 256, (yy // 7) % 256], -1) + rng.integers(-4, 5, (1500, 2000, 3)),
                 0, 255).astype(np.uint8)
    data = opng.write(px, 8, 2, filters=list(rng.integers(0, 3, 1500)))
    assert opng.parse(data) is None                                    # above the raw-size cap: left to the host
    assert np.array_equal(opng.decode(data, max_raw=None), _pillow(data))
    buf = io.BytesIO()
    Image.fromarray(px[:375, :500]).save(buf, format="PNG")            # Pillow's own filter choice
    assert np.array_equal(opng.decode(buf.getvalue()), px[:375, :500])


def _left_out():
    px = np.random.default_rng(2).integers(0, 256, (8, 8, 3)).astype(np.uint8)
    good = opng.write(px, 8, 2)
    bad_ihdr = bytearray(good)
    bad_ihdr[29] ^= 1                                                   # IHDR CRC
    dictionary = zlib.compressobj(6, zlib.DEFLATED, 15, 8, zlib.Z_DEFAULT_STRATEGY, zdict=b"abc")
    raw = opng.filter_rows(px.reshape(8, -1), [0] * 8, 3)
    bad_header = bytearray(zlib.compress(raw))
    bad_header[0] = 0x88                                                # CINFO 8
    big = np.zeros((1100, 1300, 3), np.uint8)
    return {
        "interlaced": opng.write(px, 8, 2, interlace=1),
        "apng": opng.write(px, 8, 2, before_idat=[opng.chunk(b"acTL", struct.pack(">II", 1, 0))]),
        "bad_ihdr_crc": bytes(bad_ihdr),
        "unknown_critical": opng.write(px, 8, 2, before_idat=[opng.chunk(b"ABCD", b"x")]),
        "bad_zlib_header": opng.write(px, 8, 2, zdata_override=bytes(bad_header)),
        "preset_dictionary": opng.write(px, 8, 2, zdata_override=dictionary.compress(raw) + dictionary.flush()),
        "above_cap": opng.write(big, 8, 2, level=1),
        "iccp": opng.write(px, 8, 2, before_idat=[opng.chunk(b"iCCP", b"p\0\0" + zlib.compress(b"x"))]),
        "chrm_5_bytes_before_idat": opng.write(px, 8, 2, before_idat=[opng.chunk(b"cHRM", bytes(5))]),
        "chrm_33_bytes_after_idat": opng.write(px, 8, 2, after_idat=[opng.chunk(b"cHRM", bytes(33))]),
        "not_png": b"\xff\xd8\xff\xe0" + bytes(100),
    }


def _pack(lib, datas):
    from graphnet_classifier_b200 import _lib
    n = len(datas)
    size = ctypes.sizeof(_lib.GncPngImage)
    stream = (ctypes.c_uint8 * max(1, sum(len(d) for d in datas)))()
    images = (ctypes.c_uint8 * (n * size))()
    index = (ctypes.c_int32 * n)()
    totals = (ctypes.c_int64 * 4)()
    ptrs = (ctypes.c_char_p * n)(*datas)
    sizes = (ctypes.c_int64 * n)(*[len(d) for d in datas])
    assert lib.gnc_png_pack(ctypes.cast(ptrs, ctypes.c_void_p), ctypes.cast(sizes, ctypes.c_void_p), n, 4,
                            ctypes.addressof(stream), len(stream), ctypes.addressof(images),
                            ctypes.cast(index, ctypes.c_void_p), ctypes.cast(totals, ctypes.c_void_p)) == 0
    m = int(totals[0])
    descs = ctypes.cast(images, ctypes.POINTER(_lib.GncPngImage))
    return [int(index[j]) for j in range(m)], [descs[j] for j in range(m)], bytes(stream)[:int(totals[1])], list(totals)


def test_packer_accepts_exactly_the_in_scope_files(libgnc, cases):
    left = _left_out()
    for name, data in left.items():
        assert opng.parse(data) is None, name
    datas = [d for _, d in cases] + list(left.values())
    index, descs, stream, totals = _pack(libgnc, datas)
    assert sorted(index) == list(range(len(cases)))
    assert [d.stream_bytes for d in descs] == sorted((d.stream_bytes for d in descs), reverse=True)   # longest first
    for i, d in zip(index, descs):
        ihdr, palette, z = opng.parse(datas[i])
        assert (d.width, d.height, d.bit_depth, d.color_type) == (ihdr["width"], ihdr["height"], ihdr["depth"], ihdr["color_type"])
        assert stream[d.stream_offset:d.stream_offset + d.stream_bytes] == z
        assert d.raw_bytes == ihdr["height"] * (1 + opng.row_bytes(ihdr["width"], ihdr["depth"], ihdr["color_type"]))
        assert bytes(bytearray(d.palette[k][c] for k in range(256) for c in range(3)))[:len(palette)] == palette
    assert totals[1] == sum(d.stream_bytes for d in descs) and totals[2] == sum(d.raw_bytes for d in descs)
    assert totals[3] == sum(d.width * d.height for d in descs)


def test_left_out_chunks_pillow_raises_on():
    """Chunks the packer leaves out because Pillow's reader raises on them, before and after IDAT."""
    left = _left_out()
    for name in ("chrm_5_bytes_before_idat", "chrm_33_bytes_after_idat"):
        with pytest.raises(Exception):
            _pillow(left[name])


def test_accepted_ancillary_chunks_never_make_pillow_raise(libgnc):
    """Every ancillary chunk Pillow has a reader for, at every length 0..40, before and after IDAT, in every colour
    type: whenever the packer keeps the file, Pillow decodes it to the oracle's pixels."""
    rng = np.random.default_rng(9)
    datas = []
    for ct in (0, 2, 3, 4, 6):
        px = rng.integers(0, 256, (3, 4, opng.CHANNELS[ct])).astype(np.uint8)
        pal = bytes(range(48)) if ct == 3 else None
        for ctype in (b"tRNS", b"gAMA", b"cHRM", b"sRGB", b"pHYs", b"tEXt", b"eXIf", b"bKGD", b"sBIT"):
            for n in range(41):
                body = bytes(rng.integers(0, 256, n, dtype=np.uint8))
                for where in ("before_idat", "after_idat"):
                    datas.append(opng.write(px, 8, ct, palette=pal, **{where: [opng.chunk(ctype, body)]}))
    index, _, _, _ = _pack(libgnc, datas)
    kept = set(index)
    for i, data in enumerate(datas):
        assert (i in kept) == (opng.parse(data) is not None)
        if i in kept:
            assert np.array_equal(_pillow(data), opng.decode(data))


def test_pillow_on_damaged_files():
    """The damage table of include/gnc.h: what Pillow raises on and what it accepts."""
    px = np.random.default_rng(3).integers(0, 256, (4, 5, 3)).astype(np.uint8)
    raw = opng.filter_rows(px.reshape(4, -1), [0] * 4, 3)
    z = zlib.compress(raw)
    with pytest.raises(OSError):
        _pillow(opng.write(px, 8, 2, zdata_override=z[:-1] + bytes([z[-1] ^ 1])))          # Adler-32
    with pytest.raises(OSError):
        _pillow(opng.write(px, 8, 2, raw_override=b"\x07" + raw[1:]))                     # filter type 7
    with pytest.raises(OSError):
        _pillow(opng.write(px, 8, 2, zdata_override=zlib.compress(raw[:20])))             # ends before the last row
    extra = opng.write(px, 8, 2, raw_override=raw + bytes(16))                             # data after the last row
    assert np.array_equal(_pillow(extra), px) and opng.decode(extra) is None
