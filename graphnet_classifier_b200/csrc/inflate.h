// Serial DEFLATE / zlib decoder (RFC 1950 / 1951), host + device.
//
// The PNG decoder (csrc/png.cu) runs these steps on one lane of a warp per file and lets the warp copy the matches and
// stored blocks; tests/cpu_harness/inflate_harness.cpp runs the same steps on the CPU under ASan / UBSan and compares
// them with zlib (tests/test_inflate.py).
//
// The decoder is stricter than zlib, never laxer: a stream it accepts is one zlib inflates to the same bytes.  It rejects
// block type 3, stored LEN / NLEN mismatches, code-length sets that are over-subscribed or incomplete (zlib tolerates a
// lone distance code; zlib's encoder never writes one), a missing end-of-block code, literal / length symbols 286 / 287,
// distance symbols 30 / 31, distances past the start of the output or beyond the header's window, input running out,
// output beyond `out_len` and a final block that leaves the output short.  The Adler-32 check is the caller's (the
// device computes it warp-parallel with adler_sums / adler_combine).
//
// Bounds: every read of `in` is below `in_len`, every write of `out` is below `out_len`; a Copy returned by step() lies
// inside both, so whatever the input, nothing outside the two buffers is touched.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define GNC_HD __host__ __device__ __forceinline__
#else
#define GNC_HD inline
#endif

namespace gnc {
namespace inflate {

// Per-stream status.  0 = decoded; anything else = the stream (or, for kBadFilter, the PNG rows) is not decoded.
enum : int32_t {
  kOk = 0,
  kBadHeader = 1,      // zlib header: method, window, check bits or preset dictionary
  kBadBlockType = 2,   // block type 3
  kBadStored = 3,      // stored block LEN != ~NLEN
  kBadCodes = 4,       // code-length set over-subscribed, incomplete, too many codes or no end-of-block code
  kBadSymbol = 5,      // literal / length 286, 287 or distance 30, 31
  kBadDistance = 6,    // distance past the start of the output or beyond the window
  kInputEnd = 7,       // the stream ends inside a block or the trailer
  kOverrun = 8,        // more output than out_len
  kUnderrun = 9,       // the final block ends before out_len
  kBadAdler = 10,      // Adler-32 mismatch
  kBadFilter = 11,     // PNG: a filter type byte > 4
};

constexpr int kFastBits = 10;

// Canonical Huffman code: a kFastBits-bit first-level table, and the canonical walk (puff.c) for longer codes.
struct Huffman {
  uint16_t fast[1 << kFastBits];  // (symbol << 4) | length, indexed by the next kFastBits input bits; 0 = longer code
  uint16_t count[16];             // codes of each length
  uint16_t symbol[288];           // symbols ordered by code
  uint16_t offs[16];              // build(): first index in `symbol` of each length
};

struct Bits {
  const uint8_t* in;
  uint32_t len, pos;
  uint64_t buf;
  int cnt;
  GNC_HD void refill() {
    while (cnt <= 56 && pos < len) { buf |= (uint64_t)in[pos++] << cnt; cnt += 8; }
  }
  GNC_HD bool need(int n) {
    if (cnt < n) refill();
    return cnt >= n;
  }
  GNC_HD uint32_t take(int n) {  // n <= 32, after need(n)
    const uint32_t v = (uint32_t)(buf & ((n == 32) ? 0xffffffffull : ((1ull << n) - 1)));
    buf >>= n;
    cnt -= n;
    return v;
  }
};

enum : int32_t { kModeHeader = 0, kModeCodes = 1, kModeDone = 2 };

// The decoder writes literals into a ring of kRing bytes (out[pos & (kRing - 1)]): the caller moves them to the real
// output between steps and performs each Copy on both, so that matches read the ring, never the output.
constexpr uint32_t kRing = 32768;

struct State {
  Bits br;
  uint32_t out_pos, out_len, window;
  uint32_t flush_at;  // step() also returns, with nothing to copy, when out_pos reaches this (literals to move out)
  int32_t mode, final;
  uint32_t adler;  // the trailer's Adler-32, once mode == kModeDone
};

// A copy the caller performs before the next step(): out[dst, dst + len) from out[dst - dist ..] repeating with period
// dist (a match, dist > 0), or from in[src, src + len) (a stored block, dist == 0).  len == 0: nothing to copy.
struct Copy {
  uint32_t dst, len, dist, src;
};

// zlib header (RFC 1950): method 8, CINFO <= 7, FCHECK, no preset dictionary.  window = 1 << (CINFO + 8).
GNC_HD int parse_header(const uint8_t* in, uint32_t in_len, uint32_t& window) {
  if (in_len < 2) return kInputEnd;
  const uint32_t cmf = in[0], flg = in[1];
  if ((cmf & 15) != 8 || (cmf >> 4) > 7 || ((cmf << 8) | flg) % 31 != 0 || (flg & 0x20)) return kBadHeader;
  window = 1u << ((cmf >> 4) + 8);
  return kOk;
}

GNC_HD void init(State& s, const uint8_t* in, uint32_t in_len, uint32_t out_len, uint32_t window) {
  s.br.in = in;
  s.br.len = in_len;
  s.br.pos = 2;  // after the header
  s.br.buf = 0;
  s.br.cnt = 0;
  s.out_pos = 0;
  s.out_len = out_len;
  s.window = window;
  s.flush_at = 0;
  s.mode = kModeHeader;
  s.final = 0;
  s.adler = 0;
}

GNC_HD int build(Huffman& h, const uint8_t* lens, int n) {
  for (int l = 0; l < 16; ++l) h.count[l] = 0;
  for (int s = 0; s < n; ++s) h.count[lens[s]]++;
  h.count[0] = 0;
  int left = 1;
  for (int l = 1; l < 16; ++l) {
    left = (left << 1) - h.count[l];
    if (left < 0) return kBadCodes;  // over-subscribed
  }
  if (left > 0) return kBadCodes;    // incomplete (or empty)
  h.offs[1] = 0;
  for (int l = 1; l < 15; ++l) h.offs[l + 1] = (uint16_t)(h.offs[l] + h.count[l]);
  for (int s = 0; s < n; ++s)
    if (lens[s]) h.symbol[h.offs[lens[s]]++] = (uint16_t)s;
  for (int i = 0; i < (1 << kFastBits); ++i) h.fast[i] = 0;
  uint32_t code = 0;
  int idx = 0;
  for (int l = 1; l <= kFastBits; ++l) {
    for (int k = 0; k < h.count[l]; ++k, ++idx, ++code) {
      uint32_t rev = 0;
      for (int b = 0; b < l; ++b) rev |= ((code >> b) & 1u) << (l - 1 - b);
      const uint16_t e = (uint16_t)((h.symbol[idx] << 4) | l);
      for (uint32_t j = rev; j < (1u << kFastBits); j += 1u << l) h.fast[j] = e;
    }
    code <<= 1;
  }
  return kOk;
}

// Next symbol, or -1 when the input ends inside its code.  Codes are complete, so every bit pattern decodes.
GNC_HD int decode(Bits& br, const Huffman& h) {
  if (br.cnt < 15) br.refill();
  const uint16_t e = h.fast[br.buf & ((1u << kFastBits) - 1)];
  int len, sym;
  if (e) {
    len = e & 15;
    sym = e >> 4;
  } else {
    int code = 0, first = 0, index = 0;
    sym = -1;
    for (len = 1; len < 16; ++len) {
      code |= (int)((br.buf >> (len - 1)) & 1u);
      const int count = h.count[len];
      if (code - count < first) { sym = h.symbol[index + (code - first)]; break; }
      index += count;
      first = (first + count) << 1;
      code <<= 1;
    }
    if (sym < 0) return -1;
  }
  if (len > br.cnt) return -1;
  br.buf >>= len;
  br.cnt -= len;
  return sym;
}

GNC_HD void fixed_lengths(uint8_t* lens) {
  for (int i = 0; i < 288; ++i) lens[i] = (uint8_t)(i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8);
  for (int i = 0; i < 32; ++i) lens[288 + i] = 5;
}

// Dynamic block header -> lit / dist tables (`dist` also serves as the code-length code's table).  lens: 320 bytes.
GNC_HD int read_dynamic(Bits& br, Huffman& lit, Huffman& dist, uint8_t* lens) {
  if (!br.need(14)) return kInputEnd;
  const int nlen = (int)br.take(5) + 257, ndist = (int)br.take(5) + 1, ncode = (int)br.take(4) + 4;
  if (nlen > 286 || ndist > 30) return kBadCodes;
  // the code-length code's order 16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4 | 12, 3, 13, 2, 14, 1, 15 in 5-bit fields
  const uint64_t order_lo = 0x22caa324e804a30ull, order_hi = 0x3c2e1346cull;
  for (int i = 0; i < 19; ++i) lens[i] = 0;
  for (int i = 0; i < ncode; ++i) {
    if (!br.need(3)) return kInputEnd;
    lens[(i < 12 ? order_lo >> (5 * i) : order_hi >> (5 * (i - 12))) & 31] = (uint8_t)br.take(3);
  }
  if (int rc = build(dist, lens, 19)) return rc;
  int i = 0;
  while (i < nlen + ndist) {
    const int sym = decode(br, dist);
    if (sym < 0) return kInputEnd;
    if (sym < 16) { lens[i++] = (uint8_t)sym; continue; }
    int rep;
    uint8_t val = 0;
    if (sym == 16) {
      if (i == 0) return kBadCodes;
      val = lens[i - 1];
      if (!br.need(2)) return kInputEnd;
      rep = 3 + (int)br.take(2);
    } else if (sym == 17) {
      if (!br.need(3)) return kInputEnd;
      rep = 3 + (int)br.take(3);
    } else {
      if (!br.need(7)) return kInputEnd;
      rep = 11 + (int)br.take(7);
    }
    if (i + rep > nlen + ndist) return kBadCodes;
    while (rep--) lens[i++] = val;
  }
  if (lens[256] == 0) return kBadCodes;  // no end-of-block code
  if (int rc = build(lit, lens, nlen)) return rc;
  return build(dist, lens + nlen, ndist);
}

// Decodes until the next copy, s.flush_at, the end of the stream or an error.  Literals are written to ring[out_pos %
// kRing] here.  Returns a status; with kOk, c.len > 0 (perform the copy, then call again), s.mode == kModeDone (trailer
// read into s.adler) or neither (out_pos reached flush_at: move the literals out, then call again).
GNC_HD int step(State& s, Huffman& lit, Huffman& dist, uint8_t* lens, uint8_t* ring, Copy& c) {
  c.len = 0;
  Bits& br = s.br;
  for (;;) {
    if (s.mode == kModeDone) return kOk;
    if (s.mode == kModeHeader) {
      if (s.final) {  // trailer: byte-aligned big-endian Adler-32
        br.take(br.cnt & 7);
        if (!br.need(32)) return kInputEnd;
        const uint32_t v = br.take(32);
        s.adler = (v >> 24) | ((v >> 8) & 0xff00u) | ((v << 8) & 0xff0000u) | (v << 24);
        s.mode = kModeDone;
        return s.out_pos == s.out_len ? kOk : kUnderrun;
      }
      if (!br.need(3)) return kInputEnd;
      s.final = (int32_t)br.take(1);
      const uint32_t type = br.take(2);
      if (type == 0) {
        br.take(br.cnt & 7);
        if (!br.need(32)) return kInputEnd;
        const uint32_t ln = br.take(16), nln = br.take(16);
        if (ln != (~nln & 0xffffu)) return kBadStored;
        br.pos -= (uint32_t)(br.cnt >> 3);  // hand the read-ahead bytes back: the block's bytes start at pos
        br.buf = 0;
        br.cnt = 0;
        if (ln > br.len - br.pos) return kInputEnd;
        if (ln > s.out_len - s.out_pos) return kOverrun;
        if (ln == 0) continue;
        c.dst = s.out_pos; c.len = ln; c.dist = 0; c.src = br.pos;
        br.pos += ln;
        s.out_pos += ln;
        return kOk;
      }
      if (type == 3) return kBadBlockType;
      if (type == 1) {
        fixed_lengths(lens);
        build(lit, lens, 288);
        build(dist, lens + 288, 32);
      } else if (int rc = read_dynamic(br, lit, dist, lens)) {
        return rc;
      }
      s.mode = kModeCodes;
    }
    for (;;) {  // kModeCodes
      br.refill();
      const int sym = decode(br, lit);
      if (sym < 0) return kInputEnd;
      if (sym < 256) {
        if (s.out_pos >= s.out_len) return kOverrun;
        ring[s.out_pos++ & (kRing - 1)] = (uint8_t)sym;
        if (s.out_pos == s.flush_at) return kOk;
        continue;
      }
      if (sym == 256) { s.mode = kModeHeader; break; }
      if (sym > 285) return kBadSymbol;
      const int lc = sym - 257;
      uint32_t length;
      if (lc < 8) length = 3 + lc;
      else if (lc == 28) length = 258;
      else {
        const int eb = (lc - 4) >> 2;
        if (!br.need(eb)) return kInputEnd;
        length = ((4u + (lc & 3)) << eb) + 3 + br.take(eb);
      }
      const int dc = decode(br, dist);
      if (dc < 0) return kInputEnd;
      if (dc > 29) return kBadSymbol;
      uint32_t d;
      if (dc < 4) d = 1 + dc;
      else {
        const int eb = (dc - 2) >> 1;
        if (!br.need(eb)) return kInputEnd;
        d = ((2u + (dc & 1)) << eb) + 1 + br.take(eb);
      }
      if (d > s.out_pos || d > s.window) return kBadDistance;
      if (length > s.out_len - s.out_pos) return kOverrun;
      c.dst = s.out_pos; c.len = length; c.dist = d; c.src = 0;
      s.out_pos += length;
      return kOk;
    }
  }
}

// Adler-32 sums of a byte range taken from zero: s1 = sum of bytes, s2 = sum of the running s1 after each byte, both mod
// 65521.  adler32(x) = ((n + s2) % 65521) << 16 | (1 + s1) % 65521.
GNC_HD void adler_sums(const uint8_t* p, uint64_t n, uint32_t& s1, uint32_t& s2) {
  uint64_t a = 0, b = 0;
  while (n > 0) {
    const uint64_t k = n < 4096 ? n : 4096;
    for (uint64_t i = 0; i < k; ++i) { a += p[i]; b += a; }
    a %= 65521u; b %= 65521u;
    p += k; n -= k;
  }
  s1 = (uint32_t)a; s2 = (uint32_t)b;
}

// Sums of X followed by Y (Y has ny bytes).
GNC_HD void adler_combine(uint32_t& s1x, uint32_t& s2x, uint32_t s1y, uint32_t s2y, uint64_t ny) {
  s2x = (uint32_t)((s2x + (ny % 65521u) * s1x + s2y) % 65521u);
  s1x = (s1x + s1y) % 65521u;
}

GNC_HD uint32_t adler_value(uint32_t s1, uint32_t s2, uint64_t n) {
  return (uint32_t)(((n % 65521u + s2) % 65521u) << 16) | ((1u + s1) % 65521u);
}

}  // namespace inflate
}  // namespace gnc
