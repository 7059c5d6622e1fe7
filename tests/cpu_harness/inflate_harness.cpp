// CPU harness: runs the host+device DEFLATE steps of graphnet_classifier_b200/csrc/inflate.h the way png_inflate_kernel
// does (steps into the 32 KB ring, literals moved out and copies done on ring and output, then Adler-32 from segment
// sums) so that tests/test_inflate.py can
// compare them with zlib under -fsanitize=address,undefined.  Test code only.
//
// stdin: records  [u32 stream bytes][u32 output bytes][stream]  until EOF.
// stdout: per record  [i32 status][output bytes when the status is 0].
// Every stream and output buffer is allocated at its exact size, so a read or write past either one is an ASan error.
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "../../graphnet_classifier_b200/csrc/inflate.h"

namespace inf = gnc::inflate;

static const uint32_t kFlush = 8192;  // as png_inflate_kernel: literals move out of the ring at least every kFlush bytes

static int run(const uint8_t* in, uint32_t in_len, uint8_t* out, uint32_t out_len) {
  uint32_t window = 0;
  if (int rc = inf::parse_header(in, in_len, window)) return rc;
  inf::State s;
  inf::init(s, in, in_len, out_len, window);
  auto* lit = new inf::Huffman;
  auto* dist = new inf::Huffman;
  auto* lens = new uint8_t[320];
  auto* ring = new uint8_t[inf::kRing];
  const uint32_t mask = inf::kRing - 1;
  uint32_t flushed = 0;
  int st;
  for (;;) {
    inf::Copy c;
    s.flush_at = s.out_pos + kFlush;
    st = inf::step(s, *lit, *dist, lens, ring, c);
    const uint32_t lit_end = c.len ? c.dst : s.out_pos;
    for (uint32_t i = flushed; i < lit_end && st == inf::kOk; ++i) out[i] = ring[i & mask];
    if (st != inf::kOk || s.mode == inf::kModeDone) break;
    for (uint32_t i = 0; i < c.len; ++i) {
      const uint8_t v = c.dist ? ring[(c.dst - c.dist + (i < c.dist ? i : i % c.dist)) & mask] : in[c.src + i];
      ring[(c.dst + i) & mask] = v;
      out[c.dst + i] = v;
    }
    flushed = c.len ? c.dst + c.len : s.out_pos;
  }
  delete lit; delete dist; delete[] lens; delete[] ring;
  if (st != inf::kOk) return st;
  // Adler-32 as the kernel forms it: 32 segments, summed and combined
  const uint32_t seg = (out_len + 31) / 32;
  uint32_t a1 = 0, a2 = 0;
  for (uint32_t k = 0; k < 32; ++k) {
    const uint32_t lo = k * seg < out_len ? k * seg : out_len, hi = lo + seg < out_len ? lo + seg : out_len;
    uint32_t s1, s2;
    inf::adler_sums(out + lo, hi - lo, s1, s2);
    inf::adler_combine(a1, a2, s1, s2, hi - lo);
  }
  return inf::adler_value(a1, a2, out_len) == s.adler ? inf::kOk : inf::kBadAdler;
}

int main() {
  uint32_t hdr[2];
  while (fread(hdr, 4, 2, stdin) == 2) {
    std::vector<uint8_t> tmp(hdr[0]);
    if (hdr[0] && fread(tmp.data(), 1, hdr[0], stdin) != hdr[0]) return 2;
    uint8_t* in = new uint8_t[hdr[0]];
    if (hdr[0]) memcpy(in, tmp.data(), hdr[0]);
    uint8_t* out = new uint8_t[hdr[1]];
    const int32_t st = run(in, hdr[0], out, hdr[1]);
    fwrite(&st, 4, 1, stdout);
    if (st == 0 && hdr[1]) fwrite(out, 1, hdr[1], stdout);
    delete[] in;
    delete[] out;
  }
  return 0;
}
