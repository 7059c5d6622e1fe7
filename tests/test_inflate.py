"""CPU: the shared DEFLATE decoder (csrc/inflate.h, run by tests/cpu_harness/inflate_harness.cpp under ASan / UBSan)
against zlib: every stream the encoder writes decodes to zlib's bytes, and a damaged stream is either rejected or
decoded to exactly what zlib decodes it to, with a matching Adler-32."""
import os
import struct
import subprocess
import tempfile
import zlib

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings, strategies as st

HERE = os.path.dirname(os.path.abspath(__file__))
OK, BAD_HEADER, BAD_BLOCK_TYPE, BAD_STORED, BAD_CODES, BAD_SYMBOL, BAD_DISTANCE, INPUT_END, OVERRUN, UNDERRUN, BAD_ADLER = range(11)


@pytest.fixture(scope="module")
def harness():
    exe = os.path.join(tempfile.gettempdir(), f"gnc_inflate_harness_{os.getuid()}")
    src = os.path.join(HERE, "cpu_harness", "inflate_harness.cpp")
    subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                           "-o", exe, src])

    def run(cases):
        """[(stream, out_len)] -> [(status, bytes or None)]; a sanitizer report fails the run."""
        blob = b"".join(struct.pack("<II", len(s), n) + s for s, n in cases)
        res = subprocess.run([exe], input=blob, capture_output=True,
                             env=dict(os.environ, ASAN_OPTIONS="detect_leaks=1:abort_on_error=0"))
        assert res.returncode == 0 and not res.stderr, res.stderr.decode(errors="replace")[-4000:]
        out, pos = [], 0
        for _, n in cases:
            status = struct.unpack_from("<i", res.stdout, pos)[0]
            pos += 4
            if status == OK:
                out.append((status, res.stdout[pos:pos + n]))
                pos += n
            else:
                out.append((status, None))
        assert pos == len(res.stdout)
        return out

    return run


def _payloads():
    rng = np.random.default_rng(0)
    smooth = (np.add.outer(np.arange(300), np.arange(400)) // 3 % 256).astype(np.uint8).tobytes()
    noise = rng.integers(0, 256, 70000, dtype=np.uint8).tobytes()
    runs = bytes(rng.integers(0, 4, 5000, dtype=np.uint8).repeat(7))
    return [b"\x00", b"abc" * 1000, smooth, noise, runs, bytes(range(256)) * 300, b"\x00" * 100000,
            smooth[:40000] + noise[:30000] + smooth[:40000]]


ENCODINGS = [(level, strategy, wbits) for level in (0, 1, 6, 9)
             for strategy in (zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED)
             for wbits in (9, 12, 15)]


def _compress(data, level, strategy, wbits):
    co = zlib.compressobj(level, zlib.DEFLATED, wbits, 8, strategy)
    return co.compress(data) + co.flush()


def test_encoder_streams_decode_to_zlibs_bytes(harness):
    cases = [(_compress(p, *enc), len(p)) for p in _payloads() for enc in ENCODINGS]
    for (stream, n), (status, out) in zip(cases, harness(cases)):
        assert status == OK, (len(stream), n, status)
        assert out == zlib.decompress(stream)


def test_flushed_and_multi_block_streams(harness):
    data = b"".join(bytes([i % 251]) * (i % 17 + 1) for i in range(20000))
    co = zlib.compressobj(6, zlib.DEFLATED, 15)
    parts = []
    for k in range(0, len(data), 7000):     # sync and full flushes put empty stored blocks in the stream
        parts.append(co.compress(data[k:k + 7000]))
        parts.append(co.flush(zlib.Z_SYNC_FLUSH if k % 14000 else zlib.Z_FULL_FLUSH))
    stream = b"".join(parts) + co.flush()
    [(status, out)] = harness([(stream, len(data))])
    assert status == OK and out == data


def test_rejections(harness):
    data = (bytes(range(256)) + bytes(44)) * 40   # repeats 300 bytes back
    good = zlib.compress(data, 9)
    bad_adler = good[:-1] + bytes([good[-1] ^ 1])
    far = bytearray(good)
    far[0] = 0x08                                  # CINFO 0: a 256-byte window, but the stream reaches 300 back
    far[1] = (31 - ((0x08 << 8) % 31)) % 31
    dictionary = zlib.compressobj(6, zlib.DEFLATED, 15, 8, zlib.Z_DEFAULT_STRATEGY, zdict=b"abc")
    with_dict = dictionary.compress(data) + dictionary.flush()
    stored = bytearray(_compress(data[:100], 0, zlib.Z_DEFAULT_STRATEGY, 15))
    stored[5] ^= 0xff                              # NLEN no longer ~LEN
    type3 = bytes([0x78, 0x9c, 0x07])              # final block of type 3
    cases = {
        BAD_ADLER: (bad_adler, len(data)),
        BAD_DISTANCE: (bytes(far), len(data)),
        BAD_HEADER: (with_dict, len(data)),
        BAD_STORED: (bytes(stored), 100),
        BAD_BLOCK_TYPE: (type3, 10),
        INPUT_END: (good[:len(good) // 2], len(data)),
        OVERRUN: (good, len(data) - 1),
        UNDERRUN: (good, len(data) + 1),
    }
    results = harness(list(cases.values()))
    for (expected, _), (status, _) in zip(cases.items(), results):
        assert status == expected


class BitWriter:
    """DEFLATE bit packing: fields LSB first, Huffman codes most significant bit first."""

    def __init__(self):
        self.bits = []

    def field(self, value, n):
        self.bits += [(value >> k) & 1 for k in range(n)]
        return self

    def code(self, code, n):
        self.bits += [(code >> (n - 1 - k)) & 1 for k in range(n)]
        return self

    def zlib(self):
        bits = self.bits + [0] * (-len(self.bits) % 8)
        body = bytes(sum(bits[i + k] << k for k in range(8)) for i in range(0, len(bits), 8))
        return bytes([0x78, 0x9c]) + body + bytes(4)


def _fixed_literal(w, sym):
    return w.code(0x30 + sym, 8) if sym < 144 else w.code(0x190 + sym - 144, 9)


def _dynamic(lit_lens, dist_lens):
    """A final dynamic block header whose code-length code gives symbols 0..15 four bits each (complete), followed by
    the given literal / length and distance code lengths."""
    w = BitWriter().field(1, 1).field(2, 2)
    w.field(len(lit_lens) - 257, 5).field(len(dist_lens) - 1, 5).field(19 - 4, 4)
    order = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
    for sym in order:
        w.field(0 if sym >= 16 else 4, 3)
    for n in list(lit_lens) + list(dist_lens):
        w.code(n, 4)
    return w


def _lens(n, **at):
    out = [0] * n
    for k, v in at.items():
        out[int(k[1:])] = v
    return out


def test_hand_made_rejections(harness):
    """Each rejection of csrc/inflate.h on a stream built for it, with the status it must give."""
    fixed = lambda: BitWriter().field(1, 1).field(1, 2)
    cases = {
        "literal 286": (fixed().code(0xc0 + 286 - 280, 8), BAD_SYMBOL),
        "literal 287": (fixed().code(0xc0 + 287 - 280, 8), BAD_SYMBOL),
        "distance 30": (_fixed_literal(fixed(), 97).code(1, 7).code(30, 5), BAD_SYMBOL),
        "distance 31": (_fixed_literal(fixed(), 97).code(1, 7).code(31, 5), BAD_SYMBOL),
        "distance before the output": (_fixed_literal(fixed(), 97).code(1, 7).code(1, 5), BAD_DISTANCE),
        "distance at the start": (fixed().code(1, 7).code(0, 5), BAD_DISTANCE),
        "incomplete literal set": (_dynamic(_lens(257, s0=2, s65=2, s256=2), [1, 1]), BAD_CODES),
        "over-subscribed literal set": (_dynamic(_lens(257, s0=1, s65=1, s256=1), [1, 1]), BAD_CODES),
        "lone distance code": (_dynamic(_lens(257, s0=1, s256=1), [1]), BAD_CODES),
        "over-subscribed distance set": (_dynamic(_lens(257, s0=1, s256=1), [1, 1, 1]), BAD_CODES),
        "no end-of-block code": (_dynamic(_lens(257, s0=1, s1=1), [1, 1]), BAD_CODES),
        "30 literal / length codes too many": (_dynamic(_lens(287, s0=1, s256=1), [1, 1]), BAD_CODES),
    }
    # code-length codes: all nineteen at one bit (over-subscribed), one at one bit (incomplete)
    over = BitWriter().field(1, 1).field(2, 2).field(0, 5).field(0, 5).field(15, 4)
    for _ in range(19):
        over.field(1, 3)
    lone = BitWriter().field(1, 1).field(2, 2).field(0, 5).field(0, 5).field(15, 4)
    for k in range(19):
        lone.field(1 if k == 3 else 0, 3)
    cases["over-subscribed code-length code"] = (over, BAD_CODES)
    cases["incomplete code-length code"] = (lone, BAD_CODES)
    results = harness([(w.zlib(), 16) for w, _ in cases.values()])
    for (name, (_, expected)), (status, _) in zip(cases.items(), results):
        assert status == expected, (name, status)
    # the same builders make streams zlib accepts when nothing is wrong: a literal, a match of distance 1, end of block
    ok = _fixed_literal(fixed(), 97).code(1, 7).code(0, 5).code(0, 7)
    stream = ok.zlib()[:-4] + zlib.adler32(b"aaaa").to_bytes(4, "big")
    assert zlib.decompress(stream) == b"aaaa"
    assert harness([(stream, 4)]) == [(OK, b"aaaa")]


def _zlib_accepts(stream, n):
    d = zlib.decompressobj()
    try:
        out = d.decompress(stream)
    except zlib.error:
        return None
    return out if d.eof and len(out) == n else None


STREAMS = [(_compress(p, *enc), len(p)) for p in _payloads()[:6] for enc in ENCODINGS[::7]]


@settings(max_examples=60, deadline=None, suppress_health_check=[HealthCheck.too_slow])
@given(st.lists(st.tuples(st.integers(0, len(STREAMS) - 1), st.integers(0, 2), st.integers(0, 1 << 30),
                          st.integers(1, 255)), min_size=40, max_size=40))
def test_damaged_streams_never_accepted_laxly(harness, edits):
    cases = []
    for which, kind, where, value in edits:
        stream, n = STREAMS[which]
        s = bytearray(stream)
        k = where % len(s)
        if kind == 0:
            s[k] ^= value                          # flip bits
        elif kind == 1:
            del s[k:]                              # truncate
        else:
            s += bytes([value]) * (1 + where % 9)  # extend
        cases.append((bytes(s), n))
    for (stream, n), (status, out) in zip(cases, harness(cases)):
        if status == OK:
            ref = _zlib_accepts(stream, n)
            assert ref is not None and out == ref
