"""Progressive JPEG on the CPU: the restatement of libjpeg's progressive decode (oracle/jpeg_progressive.py)
against Pillow, and the host half of the device decoder (gnc_jpeg_pack_progressive in csrc/jpeg.cu, called through
libgnc without a GPU): scans, chains, frame descriptors, and the files it leaves to the host - the same files the
oracle calls Unsupported."""
import ctypes
import io

import numpy as np
import pytest
from PIL import Image

from oracle.jpeg import Unsupported
from oracle.jpeg_progressive import decode_progressive, parse_progressive


def _jpeg(rng, h, w, gray=False, noise=12, **kw):
    """tests/test_gpu_jpeg.py's recipe: smooth content plus noise; saved progressive unless told otherwise."""
    low = rng.integers(0, 256, (h // 6 + 2, w // 6 + 2, 3), dtype=np.uint8)
    arr = np.asarray(Image.fromarray(low).resize((w, h), Image.BICUBIC)).astype(int)
    arr = np.clip(arr + rng.integers(-noise, noise + 1, (h, w, 3)), 0, 255).astype(np.uint8)
    im = Image.fromarray(arr)
    if gray:
        im = im.convert("L")
    kw.setdefault("progressive", True)
    buf = io.BytesIO()
    im.save(buf, format="JPEG", **kw)
    return buf.getvalue()


def sos_segments(data: bytes):
    """[start, end) of every SOS marker segment together with its entropy-coded data."""
    out, pos = [], 2
    while pos + 4 <= len(data) and data[pos + 1] != 0xD9:
        n = (data[pos + 2] << 8) | data[pos + 3]
        if data[pos + 1] != 0xDA:
            pos += 2 + n
            continue
        e = pos + 2 + n
        while not (data[e] == 0xFF and data[e + 1] != 0 and not 0xD0 <= data[e + 1] <= 0xD7):
            e += 1
        out.append((pos, e))
        pos = e
    return out


def without_scan(data: bytes, k: int) -> bytes:
    s, e = sos_segments(data)[k]
    return data[:s] + data[e:]


def pillow(data: bytes) -> np.ndarray:
    return np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))


def left_out_files():
    """Files the progressive decoder leaves to the host, by name."""
    rng = np.random.default_rng(21)
    col = _jpeg(rng, 37, 53, quality=90)                 # Pillow's script: 10 scans, the DC refinement is scan 6
    arr = rng.integers(0, 256, (24, 40, 3), dtype=np.uint8)
    files = {"baseline": _jpeg(rng, 24, 40, quality=90, progressive=False)}
    buf = io.BytesIO()
    Image.fromarray(arr).save(buf, format="PNG")
    files["png"] = buf.getvalue()
    buf = io.BytesIO()
    Image.fromarray(arr).convert("CMYK").save(buf, format="JPEG", quality=90, progressive=True)
    files["cmyk"] = buf.getvalue()
    seg = sos_segments(col)
    for k in range(1, 10):
        files[f"cut_after_{k}"] = col[:seg[k][0]] + b"\xff\xd9"
    files["final_y_refinement_removed"] = without_scan(col, 9)
    a, b = seg[4], seg[5]                                # Y 6..63 first scan <-> Y 1..63 refinement
    files["refinement_before_first_scan"] = col[:a[0]] + col[b[0]:b[1]] + col[a[0]:a[1]] + col[b[1]:]
    p = seg[2][0]
    ns = col[p + 4]
    patched = bytearray(col)
    patched[p + 4 + 1 + 2 * ns + 1] = 64                 # Se of an AC scan
    files["se_above_63"] = bytes(patched)
    files["no_eoi"] = col[:-2]
    return files


def _pack(lib, datas, threads=1):
    from graphnet_classifier_b200 import _lib
    n = len(datas)
    stream = (ctypes.c_uint8 * max(1, sum(map(len, datas))))()
    frames = (_lib.GncJpegImage * n)()
    index = (ctypes.c_int32 * n)()
    scans = (_lib.GncJpegScan * (n * _lib.GNC_JPEG_MAX_SCANS))()
    chains = (_lib.GncJpegChain * (n * _lib.GNC_JPEG_MAX_SCANS))()
    tables = (_lib.GncJpegHuff * (n * _lib.GNC_JPEG_MAX_TABLES))()
    totals = (ctypes.c_int64 * 8)()
    ptrs = (ctypes.c_char_p * n)(*datas)
    sizes = (ctypes.c_int64 * n)(*map(len, datas))
    vp = lambda x: ctypes.cast(x, ctypes.c_void_p)
    rc = lib.gnc_jpeg_pack_progressive(vp(ptrs), vp(sizes), n, threads, vp(stream), len(stream), vp(frames), vp(index),
                                       vp(scans), len(scans), vp(chains), len(chains), vp(tables), len(tables), vp(totals))
    assert rc == 0, lib.gnc_last_error()
    m, n_scans, n_chains = totals[0], totals[5], totals[6]
    return dict(totals=list(totals), frames=frames[:m], index=list(index[:m]), scans=scans[:n_scans],
                chains=chains[:n_chains], stream=bytes(stream[:totals[1]]))


LAYOUTS = {"gray": dict(gray=True), "444": dict(subsampling=0), "422": dict(subsampling=1), "420": dict(subsampling=2)}


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("h,w", [(1, 1), (5, 4), (20, 3), (33, 47), (97, 121)])
def test_oracle_equals_pillow(layout, h, w):
    rng = np.random.default_rng(h * 1000 + w)
    for quality in (5, 50, 100):
        for extra in ({}, dict(restart_marker_blocks=3), dict(restart_marker_rows=1)):
            data = _jpeg(rng, h, w, quality=quality, **LAYOUTS[layout], **extra)
            assert np.array_equal(decode_progressive(data), pillow(data)), (quality, extra)


SHAPES = [(37, 53, 90), (120, 75, 60), (9, 200, 95)]


@pytest.mark.parametrize("gray,n_scans,n_chains", [(False, 10, 4), (True, 6, 2)])
def test_packer_scans_chains_and_frame(libgnc, gray, n_scans, n_chains):
    from graphnet_classifier_b200.utils.jpeg import parse
    kw = dict(gray=True) if gray else dict(subsampling=2)
    datas = [_jpeg(np.random.default_rng(i), h, w, quality=q, **kw) for i, (h, w, q) in enumerate(SHAPES)]
    p = _pack(libgnc, datas, threads=2)
    assert p["totals"][0] == 3 and p["index"] == [0, 1, 2]
    assert p["totals"][5] == 3 * n_scans and p["totals"][6] == 3 * n_chains
    assert p["stream"] == b"".join(datas)
    offs = np.cumsum([0] + [len(d) for d in datas])
    # chains: longest first across the batch, their scans together and in file order, one image each
    assert [c.bytes for c in p["chains"]] == sorted((c.bytes for c in p["chains"]), reverse=True)
    got = {i: [] for i in range(3)}
    for c in p["chains"]:
        sc = p["scans"][c.first_scan:c.first_scan + c.n_scans]
        assert c.bytes == sum(s.bytes for s in sc)
        assert len({s.image for s in sc}) == 1
        assert [s.offset for s in sc] == sorted(s.offset for s in sc)
        got[sc[0].image] += [(s.offset - offs[s.image], s.bytes, s.Ss, s.Se, s.Ah, s.Al, list(s.comp)[:s.ncomp]) for s in sc]
    for i, data in enumerate(datas):
        want = [(s["start"], s["end"] - s["start"], s["Ss"], s["Se"], s["Ah"], s["Al"], s["comps"])
                for s in parse_progressive(data)[5]]
        assert sorted(got[i]) == want
        # each segment ends where the marker segments of the file say
        assert [s[0] + s[1] for s in want] == [e for _, e in sos_segments(data)]
    # frame descriptors: what gnc_jpeg_parse gives for the same image saved as baseline
    for i, (h, w, q) in enumerate(SHAPES):
        base = parse(_jpeg(np.random.default_rng(i), h, w, quality=q, progressive=False, **kw))
        f = p["frames"][i]
        for k in ("width", "height", "ncomp", "mcu_x", "mcu_y", "n_blocks", "plane_bytes"):
            assert getattr(f, k) == getattr(base, k), k
        for c in range(f.ncomp):
            assert (f.hsamp[c], f.vsamp[c]) == (base.hsamp[c], base.vsamp[c])
            assert list(f.quant[f.qtab[c]]) == list(base.quant[base.qtab[c]])
    run = np.cumsum([0] + [f.n_blocks for f in p["frames"]])
    assert [f.block_offset for f in p["frames"]] == list(run[:3])
    assert [f.coef_offset for f in p["frames"]] == list(64 * run[:3])


def test_left_out_files(libgnc):
    files = left_out_files()
    keep = _jpeg(np.random.default_rng(1), 30, 30, quality=80)
    for name, data in files.items():
        with pytest.raises(Unsupported):
            decode_progressive(data)
        assert _pack(libgnc, [data])["totals"][0] == 0, name
    p = _pack(libgnc, list(files.values()) + [keep], threads=4)
    assert p["index"] == [len(files)]


def test_dc_refinement_removed_is_kept(libgnc):
    """Coefficients 1..9 complete, DC at half precision: libjpeg does not smooth, so the file is in scope."""
    data = without_scan(_jpeg(np.random.default_rng(21), 37, 53, quality=90), 6)
    assert np.array_equal(decode_progressive(data), pillow(data))
    p = _pack(libgnc, [data])
    assert p["totals"][0] == 1 and p["totals"][5] == 9 and p["totals"][6] == 4


def test_packer_agrees_with_oracle_on_random_files(libgnc):
    """Random layouts, sizes, restart intervals and cuts: the packer keeps exactly the files the oracle decodes."""
    rng = np.random.default_rng(33)
    datas = []
    for _ in range(24):
        kw = dict(quality=int(rng.integers(5, 101)))
        if rng.random() < 0.3:
            kw["gray"] = True
        else:
            kw["subsampling"] = int(rng.integers(0, 3))
        if rng.random() < 0.3:
            kw["restart_marker_blocks"] = int(rng.integers(1, 9))
        data = _jpeg(rng, int(rng.integers(1, 60)), int(rng.integers(1, 60)), **kw)
        segs = sos_segments(data)
        r = rng.random()
        if r < 0.25:
            data = without_scan(data, int(rng.integers(0, len(segs))))
        elif r < 0.4:
            data = data[:segs[int(rng.integers(1, len(segs)))][0]] + b"\xff\xd9"
        datas.append(data)
    want = []
    for i, data in enumerate(datas):
        try:
            decode_progressive(data)
            want.append(i)
        except Unsupported:
            pass
    assert 0 < len(want) < len(datas)
    assert _pack(libgnc, datas, threads=3)["index"] == want
