"""PNG restatement (numpy) and a test-side PNG writer.

``decode(data)`` restates what ``np.asarray(Image.open(f).convert('RGB'))`` gives with Pillow 12 for the files the device
decoder (csrc/png.cu) takes: chunk parse, ``zlib.decompressobj`` for the inflate, the five row filters and the conversion
table of include/gnc.h.  ``parse(data)`` restates gnc_png_pack's acceptance rules.  ``write(...)`` makes PNG files with
explicit per-row filter types, any zlib level / strategy / wbits, IDAT split at arbitrary byte positions and extra
chunks.  Only tests and scripts import this module.
"""
from __future__ import annotations

import struct
import zlib
from typing import Optional, Sequence

import numpy as np

SIGNATURE = b"\x89PNG\r\n\x1a\n"
CHANNELS = {0: 1, 2: 3, 3: 1, 4: 2, 6: 4}
DEPTHS = {0: (1, 2, 4, 8, 16), 2: (8, 16), 3: (1, 2, 4, 8), 4: (8, 16), 6: (8, 16)}
MAX_RAW_BYTES = 2 << 20


def chunk(ctype: bytes, body: bytes) -> bytes:
    return struct.pack(">I", len(body)) + ctype + body + struct.pack(">I", zlib.crc32(ctype + body) & 0xffffffff)


def row_bytes(width: int, depth: int, color_type: int) -> int:
    return (width * CHANNELS[color_type] * depth + 7) // 8


def _bpp(depth: int, color_type: int) -> int:
    return max(1, CHANNELS[color_type] * depth // 8)


def _paeth(a: int, b: int, c: int) -> int:
    p = a + b - c
    pa, pb, pc = abs(p - a), abs(p - b), abs(p - c)
    return a if (pa <= pb and pa <= pc) else (b if pb <= pc else c)


def filter_rows(rows: np.ndarray, filters: Sequence[int], bpp: int) -> bytes:
    """rows uint8 [H, row_bytes] (unfiltered) -> the filtered stream, row y filtered with filters[y]."""
    out = bytearray()
    prev = np.zeros(rows.shape[1], np.int32)
    for y, f in enumerate(filters):
        x = rows[y].astype(np.int32)
        left = np.concatenate([np.zeros(bpp, np.int32), x[:-bpp]]) if x.size > bpp else np.zeros_like(x)
        upleft = np.concatenate([np.zeros(bpp, np.int32), prev[:-bpp]]) if x.size > bpp else np.zeros_like(x)
        if f == 0:
            r = x
        elif f == 1:
            r = x - left
        elif f == 2:
            r = x - prev
        elif f == 3:
            r = x - (left + prev) // 2
        else:
            r = x - np.array([_paeth(a, b, c) for a, b, c in zip(left, prev, upleft)], np.int32)
        out.append(f)
        out += (r & 0xff).astype(np.uint8).tobytes()
        prev = x
    return bytes(out)


def unfilter(data: bytes, height: int, rb: int, bpp: int) -> np.ndarray:
    rows = np.zeros((height, rb), np.uint8)
    prev = np.zeros(rb, np.int32)
    for y in range(height):
        f = data[y * (rb + 1)]
        if f > 4:
            raise ValueError("bad filter type")
        x = np.frombuffer(data, np.uint8, rb, y * (rb + 1) + 1).astype(np.int32)
        if f == 0:
            cur = x
        elif f == 2:
            cur = (x + prev) & 0xff
        elif f == 1:
            cur = np.zeros(rb, np.int32)
            for c in range(bpp):
                cur[c::bpp] = np.cumsum(x[c::bpp]) & 0xff
        else:
            cur, up = x.tolist(), prev.tolist()
            for i in range(rb):
                a = cur[i - bpp] if i >= bpp else 0
                if f == 3:
                    cur[i] = (cur[i] + ((a + up[i]) >> 1)) & 0xff
                else:
                    cur[i] = (cur[i] + _paeth(a, up[i], up[i - bpp] if i >= bpp else 0)) & 0xff
            cur = np.array(cur, np.int32)
        rows[y] = cur
        prev = cur
    return rows


def to_rgb(rows: np.ndarray, width: int, depth: int, color_type: int, palette: bytes) -> np.ndarray:
    """Unfiltered rows -> [H, W, 3] by the conversion table of include/gnc.h."""
    h = rows.shape[0]
    if depth < 8:
        bits = np.unpackbits(rows, axis=1).reshape(h, -1, depth)[:, :width]
        v = np.zeros((h, width), np.int32)
        for k in range(depth):
            v = (v << 1) | bits[:, :, k]
        if color_type == 3:
            pal = np.zeros(768, np.uint8)
            pal[:len(palette)] = np.frombuffer(palette, np.uint8)
            return pal.reshape(256, 3)[v].astype(np.uint8)
        g = (v * {1: 255, 2: 85, 4: 17}[depth]).astype(np.uint8)
        return np.repeat(g[:, :, None], 3, axis=2)
    ch = CHANNELS[color_type]
    if depth == 8:
        px = rows[:, :width * ch].reshape(h, width, ch)
        if color_type == 3:
            pal = np.zeros(768, np.uint8)
            pal[:len(palette)] = np.frombuffer(palette, np.uint8)
            return pal.reshape(256, 3)[px[:, :, 0]]
        if color_type in (0, 4):
            return np.repeat(px[:, :, :1], 3, axis=2)
        return px[:, :, :3].copy()
    px = rows[:, :width * ch * 2].reshape(h, width, ch, 2)
    if color_type == 0:
        v = px[:, :, 0, 0].astype(np.int32) * 256 + px[:, :, 0, 1]
        g = np.minimum(v, 255).astype(np.uint8)
        return np.repeat(g[:, :, None], 3, axis=2)
    if color_type == 4:
        return np.repeat(px[:, :, :1, 0], 3, axis=2)
    return px[:, :, :3, 0].copy()


def parse(data: bytes, max_raw: Optional[int] = MAX_RAW_BYTES):
    """-> (ihdr dict, palette bytes, zlib stream) with the packer's acceptance rules, or None when the device leaves the
    file to the host.  max_raw=None: no size cap."""
    if data[:8] != SIGNATURE:
        return None
    pos, first, idat_state, plte, stream, text = 8, True, 0, None, bytearray(), 0
    ihdr = None
    while True:
        if pos == len(data) and idat_state:
            break
        if len(data) - pos < 12:
            return None
        n = struct.unpack(">I", data[pos:pos + 4])[0]
        ctype, body = data[pos + 4:pos + 8], data[pos + 8:pos + 8 + n]
        if n > 0x7fffffff or n > len(data) - pos - 12 or not ctype.isalpha() or not ctype.isascii():
            return None
        crc = struct.unpack(">I", data[pos + 8 + n:pos + 12 + n])[0]
        if ctype != b"IDAT" and zlib.crc32(ctype + body) & 0xffffffff != crc:
            return None
        if first:
            first = False
            if ctype != b"IHDR" or n != 13:
                return None
            w, h, depth, ct, comp, filt, inter = struct.unpack(">IIBBBBB", body)
            if w == 0 or h == 0 or w > 0x7fffffff or h > 0x7fffffff or comp or filt or inter:
                return None
            if depth not in DEPTHS.get(ct, ()):
                return None
            if max_raw is not None and h * (1 + row_bytes(w, depth, ct)) > max_raw:
                return None
            ihdr = dict(width=w, height=h, depth=depth, color_type=ct)
        elif ctype == b"IDAT":
            if idat_state == 2:
                return None
            idat_state = 1
            stream += body
        else:
            if idat_state == 1:
                idat_state = 2
            if ctype == b"IEND":
                if idat_state != 2:
                    return None
                break
            ct = ihdr["color_type"]
            if ctype == b"PLTE":
                if idat_state or plte is not None or ct not in (2, 3, 6) or n % 3 or n > 768:
                    return None
                plte = body
            elif not ctype[0] & 0x20:
                return None
            elif ctype in (b"acTL", b"fcTL", b"fdAT", b"iCCP", b"zTXt", b"iTXt"):
                return None
            elif ctype == b"tEXt":
                text += n
                if text > 1 << 20:
                    return None
            elif ctype == b"tRNS" and ((ct == 0 and n < 2) or (ct == 2 and n < 6)):
                return None
            elif ((ctype == b"gAMA" and n < 4) or (ctype == b"sRGB" and n < 1) or (ctype == b"pHYs" and n < 9) or
                  (ctype == b"cHRM" and n % 4)):
                return None
        pos += 12 + n
    if len(stream) < 2 or len(stream) > 0x3fffffff:
        return None
    cmf, flg = stream[0], stream[1]
    if cmf & 15 != 8 or cmf >> 4 > 7 or ((cmf << 8) | flg) % 31 or flg & 0x20:
        return None
    return ihdr, (plte or b"") if ihdr["color_type"] == 3 else b"", bytes(stream)


def decode(data: bytes, max_raw: Optional[int] = MAX_RAW_BYTES) -> Optional[np.ndarray]:
    """[H, W, 3] uint8 for the files the device decoder claims, else None (left to the host, or damaged).  With
    max_raw=None, also the in-scope files above the size cap.  Not restated: the device's stricter stream rules that
    zlib does not share (distances past the header's window, incomplete code sets); tests/test_inflate.py checks those
    on the shared decoder itself."""
    p = parse(data, max_raw)
    if p is None:
        return None
    ihdr, palette, stream = p
    w, h, depth, ct = ihdr["width"], ihdr["height"], ihdr["depth"], ihdr["color_type"]
    rb = row_bytes(w, depth, ct)
    d = zlib.decompressobj()
    try:
        raw = d.decompress(stream)
    except zlib.error:
        return None
    if not d.eof or len(raw) != h * (1 + rb):
        return None
    try:
        rows = unfilter(raw, h, rb, _bpp(depth, ct))
    except ValueError:
        return None
    return to_rgb(rows, w, depth, ct, palette)


def write(pixels: np.ndarray, depth: int, color_type: int, *, filters=None, level: int = 6,
          strategy: int = zlib.Z_DEFAULT_STRATEGY, wbits: int = 15, split: Sequence[int] = (), palette: bytes = None,
          before_idat: Sequence[bytes] = (), after_idat: Sequence[bytes] = (), iend: bool = True,
          interlace: int = 0, raw_override: bytes = None, zdata_override: bytes = None) -> bytes:
    """pixels: samples [H, W, channels] (uint8 or uint16, values within the depth) -> PNG bytes.  filters: one filter type
    per row (default 0); split: byte positions at which the zlib stream is cut into IDAT chunks; before_idat /
    after_idat: whole extra chunks (see chunk()); raw_override / zdata_override replace the filtered data / zlib stream."""
    pixels = np.asarray(pixels)
    if pixels.ndim == 2:
        pixels = pixels[:, :, None]
    h, w, ch = pixels.shape
    assert ch == CHANNELS[color_type]
    if depth < 8:
        v = pixels[:, :, 0].astype(np.uint8)
        bits = np.unpackbits(v[:, :, None], axis=2)[:, :, 8 - depth:]
        rows = np.packbits(bits.reshape(h, -1), axis=1)
    elif depth == 8:
        rows = pixels.astype(np.uint8).reshape(h, -1)
    else:
        rows = pixels.astype(">u2").view(np.uint8).reshape(h, -1)
    filters = [0] * h if filters is None else list(filters)
    raw = raw_override if raw_override is not None else filter_rows(rows, filters, _bpp(depth, color_type))
    if zdata_override is not None:
        z = zdata_override
    else:
        co = zlib.compressobj(level, zlib.DEFLATED, wbits, 8, strategy)
        z = co.compress(raw) + co.flush()
    cuts = [0] + sorted(split) + [len(z)]
    out = SIGNATURE + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, color_type, 0, 0, interlace))
    if palette is not None:
        out += chunk(b"PLTE", palette)
    out += b"".join(before_idat)
    out += b"".join(chunk(b"IDAT", z[a:b]) for a, b in zip(cuts[:-1], cuts[1:]))
    out += b"".join(after_idat)
    if iend:
        out += chunk(b"IEND", b"")
    return out


def _samples(rng, h, w, depth, color_type, photo=False):
    ch = CHANNELS[color_type]
    top = (1 << depth) - 1
    if photo:                                   # smooth gradients plus noise
        yy, xx = np.mgrid[0:h, 0:w]
        base = np.stack([(xx * 255 // max(w - 1, 1) + k * 40 + yy // 3) % 256 for k in range(ch)], -1)
        base = base + rng.integers(-6, 7, (h, w, ch))
        v = np.clip(base, 0, 255)
        return (v * 257 if depth == 16 else v).astype(np.uint16 if depth == 16 else np.uint8)
    return rng.integers(0, top + 1, (h, w, ch)).astype(np.uint16 if depth == 16 else np.uint8)


def matrix(seed: int = 0):
    """(name, PNG bytes) over the in-scope cases: every colour type x depth, each filter forced and mixed, every zlib
    strategy and wbits, small / odd / long-row sizes, IDAT splits, short and empty palettes, ancillary chunks."""
    rng = np.random.default_rng(seed)
    out = []
    for ct, depths in DEPTHS.items():
        for depth in depths:
            for (h, w) in ((1, 1), (1, 97), (97, 1), (13, 29)):
                px = _samples(rng, h, w, depth, ct)
                pal = bytes(rng.integers(0, 256, 3 * (1 << depth), dtype=np.uint8)) if ct == 3 else None
                for f in range(6):
                    filters = [f] * h if f < 5 else list(rng.integers(0, 5, h))
                    out.append((f"ct{ct}_d{depth}_{h}x{w}_f{f}", write(px, depth, ct, filters=filters, palette=pal)))
    px = _samples(rng, 40, 50, 8, 2, photo=True)
    for level in (0, 1, 6, 9):
        for strategy in (zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED):
            for wbits in (9, 12, 15):
                out.append((f"zlib_l{level}_s{strategy}_w{wbits}",
                            write(px, 8, 2, filters=list(rng.integers(0, 5, 40)), level=level, strategy=strategy,
                                  wbits=wbits)))
    z = zlib.compress(filter_rows(px.reshape(40, -1), [4] * 40, 3))
    out.append(("split_idat", write(px, 8, 2, filters=[4] * 40, split=[1, 2, 3, 50, 50, 51, len(z) - 4])))
    out.append(("no_iend", write(px, 8, 2, iend=False)))
    idx = rng.integers(0, 256, (30, 31, 1)).astype(np.uint8)
    out.append(("palette_short", write(idx, 8, 3, palette=bytes(range(30)))))
    out.append(("palette_empty", write(idx, 8, 3, palette=b"")))
    out.append(("palette_none", write(idx, 8, 3)))
    anc = [chunk(b"gAMA", struct.pack(">I", 45455)), chunk(b"tEXt", b"Comment\0hello"),
           chunk(b"pHYs", struct.pack(">IIB", 2835, 2835, 1)), chunk(b"sRGB", b"\0"), chunk(b"abCd", b"private")]
    out.append(("trns_palette", write(idx, 8, 3, palette=bytes(range(90)), before_idat=[chunk(b"tRNS", b"\0\x80")] + anc)))
    out.append(("trns_grey", write(_samples(rng, 9, 9, 8, 0), 8, 0, before_idat=[chunk(b"tRNS", b"\0\x05")],
                                   after_idat=anc)))
    out.append(("trns_grey16", write(_samples(rng, 9, 9, 16, 0), 16, 0, before_idat=[chunk(b"tRNS", b"\0\x05")])))
    out.append(("trns_rgb", write(_samples(rng, 9, 9, 8, 2), 8, 2, before_idat=[chunk(b"tRNS", bytes(6))])))
    out.append(("trns_rgb16", write(_samples(rng, 9, 9, 16, 2), 16, 2, before_idat=[chunk(b"tRNS", bytes(6))])))
    out.append(("long_rows", write(_samples(rng, 2, 12000, 8, 2), 8, 2, filters=[1, 4])))
    for depth in (1, 2, 4):
        for w in (3, 5, 7, 9, 15):
            out.append((f"odd_width_d{depth}_w{w}", write(_samples(rng, 5, w, depth, 0), depth, 0, filters=[1, 2, 3, 4, 0])))
    return out
