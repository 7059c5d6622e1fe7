"""TEST INFRASTRUCTURE - CPU restatement (pure Python + numpy) of the progressive JPEG decode behind the reference's
``Image.open(path).convert('RGB')`` (utils/dataloader.py:34 through ImageFolder's loader,
utils/image_to_graph/image_to_graph_optimized.py:65-68, utils/inference.py:47) for progressive (SOF2) files.

Pillow 12.2 decodes them through libjpeg-turbo 3.1.4 with the library defaults.  Restated from the published sources:
the marker rules (jdmarker.c, jdinput.c: Huffman tables and restart interval per scan, quantisation tables latched at a
component's first scan), the progression checks of jdphuff.c start_pass_phuff_decoder, the block-smoothing condition
of jdcoefct.c smoothing_ok, and jdphuff.c's four entropy procedures.  The inverse DCT, upsampling and colour stages are
the baseline ones (oracle/jpeg.py).

PINNED: ``tests/test_jpeg_progressive.py`` requires ``decode_progressive`` to reproduce Pillow's pixels bit for bit and
the device packer (csrc/jpeg.cu gnc_jpeg_pack_progressive) to keep exactly the files it decodes.
"""
from __future__ import annotations

import numpy as np

from oracle.jpeg import ZIGZAG, Unsupported, _Bits, _extend, _symbol, _upsample, idct_islow

# ---- progressive (SOF2) ----------------------------------------------------------------------------------------------
# jdmarker.c / jdinput.c / jdphuff.c: the frame layouts decode_baseline accepts, coded as several scans over one
# coefficient buffer.  Files libjpeg(-turbo) would not decode by the plain path are Unsupported (see
# parse_progressive); csrc/jpeg.cu's gnc_jpeg_pack_progressive leaves out exactly the same files.
MAX_SCANS, MAX_TABLES = 64, 32          # per file; include/gnc.h GNC_JPEG_MAX_SCANS / GNC_JPEG_MAX_TABLES


def _natural(k: int) -> int:
    return int(ZIGZAG[min(k, 63)])      # libjpeg's jpeg_natural_order has 16 extra entries, all 63


def _i16(v: int) -> int:
    return ((int(v) + 32768) & 0xFFFF) - 32768                                  # JCOEF is a short


def _entropy_end(data: bytes, pos: int) -> int:
    """The entropy-coded segment starting at ``pos`` runs to the next marker other than RSTn / a stuffed zero / fill."""
    e = pos
    while e + 1 < len(data):
        if data[e] == 0xFF and data[e + 1] != 0 and not 0xD0 <= data[e + 1] <= 0xD7 and data[e + 1] != 0xFF:
            return e
        e += 1
    raise Unsupported("scan runs past the end of the file")


def parse_progressive(data: bytes):
    """Markers of a progressive file -> ``(H, W, hs, vs, quant, scans)``.  ``quant[c]`` = component c's table as latched
    at its first scan (jdinput.c latch_quant_tables); ``scans`` = dicts with the components (frame indices), Ss, Se,
    Ah, Al, the restart interval and Huffman tables in force, and the entropy segment's [start, end)."""
    if data[:2] != b"\xff\xd8":
        raise Unsupported("no SOI")
    pos, quant, huff, dri, frame, adobe = 2, {}, {}, 0, None, -1
    latched, scans, coef_bits, used_tables = {}, [], None, set()
    while True:
        if pos + 2 > len(data):
            raise Unsupported("no EOI")
        if data[pos] != 0xFF:
            raise Unsupported("marker expected")
        m = data[pos + 1]
        if m == 0xFF:
            pos += 1
            continue
        pos += 2
        if m == 0xD9:
            break
        if m in (0xD8, 0x01) or 0xD0 <= m <= 0xD7:
            continue
        if pos + 2 > len(data):
            raise Unsupported("truncated")
        n = (data[pos] << 8) | data[pos + 1]
        if n < 2 or pos + n > len(data):
            raise Unsupported("segment beyond the file")
        seg = data[pos + 2:pos + n]
        if m == 0xC2:
            if frame is not None or len(seg) < 6 or seg[0] != 8:
                raise Unsupported("frame")
            H, W, nc = (seg[1] << 8) | seg[2], (seg[3] << 8) | seg[4], seg[5]
            if nc not in (1, 3) or H == 0 or W == 0 or len(seg) < 6 + 3 * nc:
                raise Unsupported("frame")
            comps = [(seg[6 + 3 * c], seg[7 + 3 * c] >> 4, seg[7 + 3 * c] & 15, seg[8 + 3 * c]) for c in range(nc)]
            if any(c[3] > 3 or not 1 <= c[1] <= 4 or not 1 <= c[2] <= 4 for c in comps) or len({c[0] for c in comps}) != nc:
                raise Unsupported("frame")
            frame = (H, W, comps)
            coef_bits = [[-1] * 64 for _ in range(nc)]
        elif 0xC0 <= m <= 0xCF and m not in (0xC4, 0xC8):
            raise Unsupported("not progressive Huffman")
        elif m == 0xDC:
            raise Unsupported("DNL")
        elif m == 0xC4:
            i = 0
            while i < len(seg):
                if i + 17 > len(seg):
                    raise Unsupported("DHT")
                tc, th = seg[i] >> 4, seg[i] & 15
                bits = list(seg[i + 1:i + 17])
                cnt = sum(bits)
                if tc > 1 or th > 3 or cnt > 256 or i + 17 + cnt > len(seg):
                    raise Unsupported("DHT")
                vals = list(seg[i + 17:i + 17 + cnt])
                if tc == 0 and any(v > 15 for v in vals):
                    raise Unsupported("DC symbol")
                table, code, k = {}, 0, 0
                for length in range(1, 17):
                    for _ in range(bits[length - 1]):
                        table[(length, code)] = vals[k]
                        code += 1
                        k += 1
                    if code >= (1 << length):                                  # jdhuff.c: no all-ones code
                        raise Unsupported("DHT codes")
                    code <<= 1
                huff[(tc, th)] = (table, object())                              # (table, identity of this definition)
                i += 17 + cnt
        elif m == 0xDB:
            i = 0
            while i < len(seg):
                pq, tq = seg[i] >> 4, seg[i] & 15
                if tq > 3 or pq > 1 or i + 1 + 64 * (pq + 1) > len(seg):
                    raise Unsupported("DQT")
                q = [(seg[i + 1 + 2 * k] << 8) | seg[i + 2 + 2 * k] for k in range(64)] if pq else list(seg[i + 1:i + 65])
                nat = np.zeros(64, np.int64)
                nat[ZIGZAG] = q
                quant[tq] = nat
                i += 1 + 64 * (pq + 1)
        elif m == 0xDD:
            if len(seg) < 2:
                raise Unsupported("DRI")
            dri = (seg[0] << 8) | seg[1]
        elif m == 0xEE:
            if len(seg) >= 12 and seg[:5] == b"Adobe":
                adobe = seg[11]
        elif m == 0xDA:
            if frame is None:
                raise Unsupported("scan before the frame")
            H, W, comps = frame
            nc = len(comps)
            if nc == 3:
                ids = [c[0] for c in comps]
                if adobe == 0 or (adobe < 0 and ids == [ord("R"), ord("G"), ord("B")]):
                    raise Unsupported("RGB colour space")
                if not (comps[1][1:3] == comps[2][1:3] == (1, 1) and comps[0][1:3] in ((1, 1), (2, 1), (2, 2))):
                    raise Unsupported("sampling")
            ns = seg[0] if seg else 0
            if not 1 <= ns <= nc or len(seg) < 1 + 2 * ns + 3:
                raise Unsupported("scan header")
            ids = [c[0] for c in comps]
            sc = []
            for j in range(ns):
                cid = seg[1 + 2 * j]
                if cid not in ids:
                    raise Unsupported("scan component")
                sc.append((ids.index(cid), seg[2 + 2 * j] >> 4, seg[2 + 2 * j] & 15))
            if [c for c, _, _ in sc] != sorted({c for c, _, _ in sc}):
                raise Unsupported("scan components out of frame order")
            Ss, Se, Ah, Al = seg[1 + 2 * ns], seg[2 + 2 * ns], seg[3 + 2 * ns] >> 4, seg[3 + 2 * ns] & 15
            # jdphuff.c start_pass_phuff_decoder: the checks it fails on, and the ones it only warns about
            if Ss == 0:
                if Se != 0:
                    raise Unsupported("DC scan with Se != 0")
            elif Ss > Se or Se > 63 or ns != 1:
                raise Unsupported("AC scan band / components")
            if (Ah and Al != Ah - 1) or Al > 13:
                raise Unsupported("successive approximation")
            for c, _, _ in sc:
                if Ss and coef_bits[c][0] < 0:
                    raise Unsupported("AC scan before the component's first DC scan")
                for k in range(Ss, Se + 1):
                    if (Ah == 0 and coef_bits[c][k] != -1) or (Ah and coef_bits[c][k] != Ah):
                        raise Unsupported("bogus progression")
                    coef_bits[c][k] = Al
            dc_tabs, ac_tab = [], None
            for c, td, ta in sc:
                if Ss == 0 and Ah == 0:
                    if (0, td) not in huff:
                        raise Unsupported("undefined DC table")
                    dc_tabs.append(huff[(0, td)])
                if Ss:
                    if (1, ta) not in huff:
                        raise Unsupported("undefined AC table")
                    ac_tab = huff[(1, ta)]
                if c not in latched:
                    if comps[c][3] not in quant:
                        raise Unsupported("undefined quantisation table")
                    latched[c] = quant[comps[c][3]]
            used_tables.update(t[1] for t in dc_tabs + ([ac_tab] if ac_tab else []))
            start = pos + n
            end = _entropy_end(data, start)
            scans.append(dict(comps=[c for c, _, _ in sc], Ss=Ss, Se=Se, Ah=Ah, Al=Al, dri=dri, start=start, end=end,
                              dc=[t[0] for t in dc_tabs], ac=ac_tab[0] if ac_tab else None))
            if len(scans) > MAX_SCANS or len(used_tables) > MAX_TABLES:
                raise Unsupported("too many scans or tables")
            pos = end
            continue
        pos += n
    if frame is None or not scans:
        raise Unsupported("no scan")
    # jdcoefct.c smoothing_ok (libjpeg-turbo >= 2.1, SAVED_COEFS = 10): with a DC never coded, or an AC coefficient
    # 1..9 of some component not fully refined, libjpeg smooths across blocks - out of scope
    if any(cb[0] < 0 or any(b != 0 for b in cb[1:10]) for cb in coef_bits):
        raise Unsupported("incompletely refined: libjpeg would apply block smoothing")
    H, W, comps = frame
    nc = len(comps)
    hs, vs = ([1], [1]) if nc == 1 else ([c[1] for c in comps], [c[2] for c in comps])
    return H, W, hs, vs, [latched[c] for c in range(nc)], scans


def _scan_blocks(sc, H, W, hs, vs, coefs):
    """Blocks of a scan in coding order, one list per MCU: interleaved scans walk the frame's MCUs, a single-component
    scan walks the component's own ceil(W h / 8 hmax) x ceil(H v / 8 vmax) blocks in raster order."""
    mcu_x, mcu_y = coefs[0].shape[1] // hs[0], coefs[0].shape[0] // vs[0]
    if len(sc["comps"]) > 1:
        for my in range(mcu_y):
            for mx in range(mcu_x):
                yield [(j, coefs[c][my * vs[c] + by, mx * hs[c] + bx]) for j, c in enumerate(sc["comps"])
                       for by in range(vs[c]) for bx in range(hs[c])]
        return
    c = sc["comps"][0]
    bw, bh = -(-W * hs[c] // (8 * hs[0])), -(-H * vs[c] // (8 * vs[0]))
    for by in range(bh):
        for bx in range(bw):
            yield [(0, coefs[c][by, bx])]


def _refine(br, blk, z, p1):
    """A correction bit for a nonzero coefficient that is not yet refined at this bit (jdphuff.c decode_mcu_AC_refine)."""
    if br.get(1) and (blk[z] & p1) == 0:
        blk[z] = _i16(blk[z] + p1 if blk[z] >= 0 else blk[z] - p1)


def _decode_scan(data, sc, blocks):
    """jdphuff.c's four procedures: decode_mcu_DC_first / _DC_refine / _AC_first / _AC_refine."""
    br = _Bits(data, sc["start"])
    Ss, Se, Ah, Al, dri = sc["Ss"], sc["Se"], sc["Ah"], sc["Al"], sc["dri"]
    pred, eobrun, left, p1 = [0, 0, 0], 0, dri, 1 << Al
    for mcu in blocks:
        if dri and left == 0:
            br.restart()
            pred, eobrun, left = [0, 0, 0], 0, dri
        for j, blk in mcu:
            if Ss == 0 and Ah == 0:
                s = _symbol(br, sc["dc"][j])
                pred[j] += _extend(br.get(s), s) if s else 0
                blk[0] = _i16(pred[j] << Al)
            elif Ss == 0:
                if br.get(1):
                    blk[0] = _i16(blk[0] | p1)
            elif Ah == 0:
                if eobrun:
                    eobrun -= 1
                    continue
                k = Ss
                while k <= Se:
                    rs = _symbol(br, sc["ac"])
                    r, s = rs >> 4, rs & 15
                    if s:
                        k += r
                        blk[_natural(k)] = _i16(_extend(br.get(s), s) << Al)
                    elif r == 15:
                        k += 15
                    else:
                        eobrun = (1 << r) + br.get(r) - 1
                        break
                    k += 1
            else:
                k = Ss
                if eobrun == 0:
                    while k <= Se:
                        rs = _symbol(br, sc["ac"])
                        r, s = rs >> 4, rs & 15
                        if s:
                            s = p1 if br.get(1) else -p1
                        elif r != 15:
                            eobrun = (1 << r) + br.get(r)
                            break
                        while True:                     # the zero run (and the new coefficient's place) passes over
                            z = _natural(k)             # nonzero coefficients: each takes a correction bit
                            if blk[z] != 0:
                                _refine(br, blk, z, p1)
                            else:
                                r -= 1
                                if r < 0:
                                    break
                            k += 1
                            if k > Se:
                                break
                        if s:
                            blk[_natural(k)] = s
                        k += 1
                if eobrun > 0:
                    while k <= Se:
                        z = _natural(k)
                        if blk[z] != 0:
                            _refine(br, blk, z, p1)
                        k += 1
                    eobrun -= 1
        if dri:
            left -= 1


def progressive_coefficients(data: bytes):
    """Progressive file -> ``(H, W, hs, vs, quant, coefs)``: every scan decoded into the frame's MCU-padded coefficient
    arrays ``coefs[c]`` = int64 ``[mcu_y v_c, mcu_x h_c, 64]`` (natural order), the layout decode_baseline uses."""
    H, W, hs, vs, quant, scans = parse_progressive(data)
    mcu_x, mcu_y = -(-W // (8 * hs[0])), -(-H // (8 * vs[0]))
    coefs = [np.zeros((mcu_y * vs[c], mcu_x * hs[c], 64), np.int64) for c in range(len(hs))]
    for sc in scans:
        _decode_scan(data, sc, _scan_blocks(sc, H, W, hs, vs, coefs))
    return H, W, hs, vs, quant, coefs


def decode_progressive(data: bytes) -> np.ndarray:
    """Progressive JPEG file bytes -> ``uint8 [H, W, 3]``, the pixels of ``Image.open(...).convert('RGB')``; Unsupported
    for the files libjpeg would not decode by the plain path (and the device decoder leaves to the host)."""
    H, W, hs, vs, quant, coefs = progressive_coefficients(data)
    nc = len(coefs)
    planes = []
    for c in range(nc):
        by, bx = coefs[c].shape[:2]
        px = idct_islow(coefs[c].reshape(-1, 64), quant[c]).reshape(by, bx, 8, 8)
        planes.append(px.transpose(0, 2, 1, 3).reshape(by * 8, bx * 8))
    Y = planes[0][:H, :W].astype(np.int64)
    if nc == 1:
        return np.stack([Y, Y, Y], -1).astype(np.uint8)
    hf, vf = hs[0] // hs[1], vs[0] // vs[1]
    dw, dh = -(-W * hs[1] // hs[0]), -(-H * vs[1] // vs[0])
    cb = _upsample(planes[1], dw, dh, hf, vf, W, H) - 128
    cr = _upsample(planes[2], dw, dh, hf, vf, W, H) - 128
    r = Y + ((91881 * cr + 32768) >> 16)
    g = Y + ((-22554 * cb + 32768 - 46802 * cr) >> 16)
    b = Y + ((116130 * cb + 32768) >> 16)
    return np.clip(np.stack([r, g, b], -1), 0, 255).astype(np.uint8)
