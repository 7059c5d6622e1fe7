// PNG decode on the device, bit for bit  np.asarray(Image.open(f).convert('RGB'))  with Pillow 12 (include/gnc.h).
//
//   host   gnc_png_pack           : chunk parse and validation on host threads -> one descriptor per file that is in,
//                                   IDAT payloads back to back in the pinned stream buffer, files longest stream first
//   device png_inflate_kernel     : one warp per file; lane 0 decodes symbols with csrc/inflate.h's steps (tables and a
//                                   32 KB window ring in shared memory), the warp moves literals out, copies matches
//                                   and stored blocks, then checks Adler-32
//   device png_unfilter_kernel    : one warp per file, row after row: the five filters undone in place, then the row
//                                   converted into the packed [H, W, 3] output with Pillow's mode rules
//
// The device may be stricter than Pillow, never laxer: a file it claims is one zlib inflates cleanly to exactly
// H * (1 + row bytes) bytes with a matching Adler-32 and filter bytes 0..4; every other file gets a nonzero status (or is
// left out by the packer) and is decoded by Pillow on the host.  The two stages are separate launches; fusing them
// (the inflating warp unfiltering each finished row) is not measured.
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <thread>
#include <vector>

#include "common.cuh"
#include "inflate.h"

namespace gnc {
namespace png {

namespace inf = gnc::inflate;

static uint32_t crc32(const uint8_t* p, int64_t n, uint32_t crc = 0) {
  static const struct Table {
    uint32_t t[256];
    Table() {
      for (uint32_t i = 0; i < 256; ++i) {
        uint32_t c = i;
        for (int k = 0; k < 8; ++k) c = (c & 1) ? 0xEDB88320u ^ (c >> 1) : c >> 1;
        t[i] = c;
      }
    }
  } table;
  crc = ~crc;
  for (int64_t i = 0; i < n; ++i) crc = table.t[(crc ^ p[i]) & 0xff] ^ (crc >> 8);
  return ~crc;
}

static inline uint32_t be32(const uint8_t* p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]; }

struct Segment { int64_t offset, bytes; };

static bool is_letter(uint8_t c) { return (c >= 'A' && c <= 'Z') || (c >= 'a' && c <= 'z'); }

// One file -> descriptor (geometry, palette, stream and raw sizes; offsets left 0) and its IDAT payloads.  GNC_OK or
// GNC_UNSUPPORTED.  Left out: anything but the table's colour type / depth pairs, interlaced files, APNG, unknown
// critical chunks, a CRC mismatch on any chunk but IDAT, IDATs that are not consecutive, chunks whose content Pillow may
// raise on (iCCP, zTXt, iTXt; short tRNS, gAMA, sRGB, pHYs; a cHRM that is not whole 4-byte values), a PLTE out of
// place, bytes that do not form whole chunks, a zlib header outside RFC 1950's plain form, and raw data above
// GNC_PNG_MAX_RAW_BYTES.
static int parse(const uint8_t* data, int64_t size, gnc_png_image_t* out, std::vector<Segment>& segs) {
  constexpr int UNSUP = GNC_UNSUPPORTED;
  static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', '\r', '\n', 0x1a, '\n'};
  segs.clear();
  memset(out, 0, sizeof(*out));
  if (!data || size < 8 + 25 || memcmp(data, sig, 8) != 0) return UNSUP;
  int64_t pos = 8;
  int n_chunks = 0, seen_plte = 0, idat_state = 0;   // idat_state: 0 before, 1 inside the IDAT run, 2 after it
  int64_t stream_bytes = 0, text_bytes = 0;
  for (;;) {
    if (pos == size && idat_state != 0) break;       // no IEND: Pillow stops at the end of the file
    if (size - pos < 12) return UNSUP;
    const uint32_t len = be32(data + pos);
    const uint8_t* type = data + pos + 4;
    const uint8_t* body = data + pos + 8;
    if (len > 0x7fffffffu || (int64_t)len > size - pos - 12) return UNSUP;
    for (int k = 0; k < 4; ++k)
      if (!is_letter(type[k])) return UNSUP;
    const bool idat = memcmp(type, "IDAT", 4) == 0;
    if (!idat && crc32(type, 4 + (int64_t)len) != be32(body + len)) return UNSUP;
    if (n_chunks++ == 0) {
      if (memcmp(type, "IHDR", 4) != 0 || len != 13) return UNSUP;
      const uint32_t w = be32(body), h = be32(body + 4);
      const int depth = body[8], ctype = body[9];
      if (w == 0 || h == 0 || w > 0x7fffffffu || h > 0x7fffffffu) return UNSUP;
      if (body[10] != 0 || body[11] != 0 || body[12] != 0) return UNSUP;     // compression, filter, interlace
      int channels;
      switch (ctype) {
        case 0: channels = 1; if (depth != 1 && depth != 2 && depth != 4 && depth != 8 && depth != 16) return UNSUP; break;
        case 2: channels = 3; if (depth != 8 && depth != 16) return UNSUP; break;
        case 3: channels = 1; if (depth != 1 && depth != 2 && depth != 4 && depth != 8) return UNSUP; break;
        case 4: channels = 2; if (depth != 8 && depth != 16) return UNSUP; break;
        case 6: channels = 4; if (depth != 8 && depth != 16) return UNSUP; break;
        default: return UNSUP;
      }
      const int64_t bits = (int64_t)w * channels * depth;
      const int64_t row_bytes = (bits + 7) / 8;
      const int64_t raw = (int64_t)h * (1 + row_bytes);
      if (raw > GNC_PNG_MAX_RAW_BYTES) return UNSUP;
      out->width = (int32_t)w; out->height = (int32_t)h;
      out->color_type = ctype; out->bit_depth = depth;
      out->row_bytes = (int32_t)row_bytes;
      out->bpp = std::max(1, channels * depth / 8);
      out->raw_bytes = raw;
    } else if (idat) {
      if (idat_state == 2) return UNSUP;
      idat_state = 1;
      segs.push_back({pos + 8, (int64_t)len});
      stream_bytes += len;
    } else {
      if (idat_state == 1) idat_state = 2;
      if (memcmp(type, "IEND", 4) == 0) {
        if (idat_state != 2) return UNSUP;
        break;
      }
      if (memcmp(type, "PLTE", 4) == 0) {
        if (idat_state != 0 || seen_plte++ || (out->color_type != 3 && out->color_type != 2 && out->color_type != 6) ||
            len % 3 != 0 || len > 768)
          return UNSUP;
        if (out->color_type == 3) memcpy(out->palette, body, len);
      } else if (!(type[0] & 0x20)) {
        return UNSUP;                                                   // IHDR again or an unknown critical chunk
      } else if (!memcmp(type, "acTL", 4) || !memcmp(type, "fcTL", 4) || !memcmp(type, "fdAT", 4) ||
                 !memcmp(type, "iCCP", 4) || !memcmp(type, "zTXt", 4) || !memcmp(type, "iTXt", 4)) {
        return UNSUP;
      } else if (!memcmp(type, "tEXt", 4)) {
        if ((text_bytes += len) > (1 << 20)) return UNSUP;             // far below Pillow's MAX_TEXT_MEMORY
      } else if (!memcmp(type, "tRNS", 4)) {
        if ((out->color_type == 0 && len < 2) || (out->color_type == 2 && len < 6)) return UNSUP;
      } else if ((!memcmp(type, "gAMA", 4) && len < 4) || (!memcmp(type, "sRGB", 4) && len < 1) ||
                 (!memcmp(type, "pHYs", 4) && len < 9) || (!memcmp(type, "cHRM", 4) && len % 4 != 0)) {
        return UNSUP;
      }
    }
    pos += 12 + (int64_t)len;
  }
  if (stream_bytes < 2 || stream_bytes > 0x3fffffff) return UNSUP;
  uint8_t head[2];
  int got = 0;
  for (const Segment& s : segs)
    for (int64_t k = 0; k < s.bytes && got < 2; ++k) head[got++] = data[s.offset + k];
  uint32_t window = 0;
  if (inf::parse_header(head, 2, window) != inf::kOk) return UNSUP;
  out->window = (int32_t)window;
  out->stream_bytes = stream_bytes;
  return GNC_OK;
}

constexpr int kWarps = 4;          // unfilter kernel: files per block
constexpr uint32_t kFlush = 8192;  // literals move from the ring to the output at least every kFlush bytes

struct InflateSmem {
  uint8_t ring[inf::kRing];        // the last 32 KB of output: matches read it, never global memory
  inf::Huffman lit, dist;
  uint8_t lens[320];
};

// One warp per block (38.5 KB of shared memory: five files per SM).  Lane 0 runs the steps; the warp moves literals out
// of the ring and performs each copy, reading every source of a 32-byte chunk before writing any of it (a source and a
// destination 32 KB apart share a ring slot).
__global__ void __launch_bounds__(32) png_inflate_kernel(const uint8_t* __restrict__ stream,
                                                         const gnc_png_image_t* __restrict__ images, int B,
                                                         uint8_t* __restrict__ raw, int32_t* __restrict__ status) {
  __shared__ InflateSmem sm;
  const int lane = threadIdx.x;
  const int f = blockIdx.x;
  if (f >= B) return;
  const gnc_png_image_t& im = images[f];
  const uint8_t* in = stream + im.stream_offset;
  uint8_t* out = raw + im.raw_offset;
  const uint32_t out_len = (uint32_t)im.raw_bytes, mask = inf::kRing - 1;
  inf::State s;
  if (lane == 0) inf::init(s, in, (uint32_t)im.stream_bytes, out_len, (uint32_t)im.window);
  int st = inf::kOk;
  uint32_t flushed = 0;
  for (;;) {
    inf::Copy c;
    int done = 0;
    uint32_t pos = 0;
    if (lane == 0) {
      s.flush_at = s.out_pos + kFlush;
      st = inf::step(s, sm.lit, sm.dist, sm.lens, sm.ring, c);
      done = st != inf::kOk || s.mode == inf::kModeDone;
      pos = s.out_pos;
    }
    __syncwarp();                                     // lane 0's literals are visible to the other lanes
    done = __shfl_sync(0xffffffffu, done, 0);
    const uint32_t len = __shfl_sync(0xffffffffu, c.len, 0);
    const uint32_t dst = __shfl_sync(0xffffffffu, c.dst, 0), dist = __shfl_sync(0xffffffffu, c.dist, 0);
    const uint32_t src = __shfl_sync(0xffffffffu, c.src, 0);
    pos = __shfl_sync(0xffffffffu, pos, 0);
    const uint32_t lit_end = len ? dst : pos;
    for (uint32_t i = flushed + lane; i < lit_end; i += 32) out[i] = sm.ring[i & mask];
    if (done) break;
    for (uint32_t b = 0; b < len; b += 32) {          // out[dst + i] = out[dst - dist + i mod dist]: every source precedes dst
      const uint32_t i = b + lane;
      uint8_t v = 0;
      if (i < len) v = dist ? sm.ring[(dst - dist + (i < dist ? i : i % dist)) & mask] : in[src + i];
      __syncwarp();
      if (i < len) { sm.ring[(dst + i) & mask] = v; out[dst + i] = v; }
    }
    __syncwarp();
    flushed = len ? dst + len : pos;
  }
  st = __shfl_sync(0xffffffffu, st, 0);
  __syncwarp();                                       // the output is complete before the Adler-32 reads it
  if (st == inf::kOk) {                               // Adler-32: 32 contiguous segments, combined on every lane
    const uint32_t seg = (out_len + 31) / 32;
    const uint32_t lo = min(out_len, lane * seg), hi = min(out_len, lo + seg);
    uint32_t s1, s2;
    inf::adler_sums(out + lo, hi - lo, s1, s2);
    uint32_t a1 = 0, a2 = 0;
    for (int k = 0; k < 32; ++k) {
      const uint32_t b1 = __shfl_sync(0xffffffffu, s1, k), b2 = __shfl_sync(0xffffffffu, s2, k);
      const uint32_t n = __shfl_sync(0xffffffffu, hi - lo, k);
      inf::adler_combine(a1, a2, b1, b2, n);
    }
    if (lane == 0 && inf::adler_value(a1, a2, out_len) != s.adler) st = inf::kBadAdler;
  }
  if (lane == 0) status[f] = st;
}

__device__ __forceinline__ int paeth(int a, int b, int c) {
  const int pa = abs(b - c), pb = abs(a - c), pc = abs(a + b - 2 * c);
  return (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c);
}

__global__ void __launch_bounds__(32 * kWarps, 4) png_unfilter_kernel(const gnc_png_image_t* __restrict__ images, int B,
                                                                    uint8_t* __restrict__ raw, uint8_t* __restrict__ rgb,
                                                                    int32_t* __restrict__ status) {
  __shared__ uint8_t pal[kWarps][768];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int f = blockIdx.x * kWarps + warp;
  if (f >= B) return;
  if (status[f] != inf::kOk) return;                  // warp-uniform
  // (the minimum of 4 blocks above: without it ptxas keeps this kernel near 40 registers and spills 20 bytes)
  const gnc_png_image_t& im = images[f];
  const int W = im.width, H = im.height, rb = im.row_bytes, bpp = im.bpp, ct = im.color_type, depth = im.bit_depth;
  if (ct == 3)
    for (int i = lane; i < 768; i += 32) pal[warp][i] = (&im.palette[0][0])[i];
  __syncwarp();
  uint8_t* base = raw + im.raw_offset;
  uint8_t* out = rgb + 3 * im.pixel_offset;
  const int npix = rb / bpp;
  for (int y = 0; y < H; ++y) {
    uint8_t* row = base + (int64_t)y * (rb + 1);
    uint8_t* cur = row + 1;
    const uint8_t* prev = y ? cur - (rb + 1) : nullptr;
    const int ft = row[0];
    if (ft > 4) {
      if (lane == 0) status[f] = inf::kBadFilter;
      return;
    }
    if (ft == 1) {                                    // Sub: a lane scan per byte position mod bpp
      for (int c = 0; c < bpp; ++c) {
        uint32_t carry = 0;
        for (int p0 = 0; p0 < npix; p0 += 32) {
          const int p = p0 + lane;
          uint32_t v = p < npix ? cur[p * bpp + c] : 0u;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, v, d);
            if (lane >= d) v += u;
          }
          v += carry;
          if (p < npix) cur[p * bpp + c] = (uint8_t)v;
          carry = __shfl_sync(0xffffffffu, v, 31);
        }
      }
    } else if (ft == 2) {                             // Up
      if (prev)
        for (int i = lane; i < rb; i += 32) cur[i] = (uint8_t)(cur[i] + prev[i]);
    } else if (ft >= 3 && lane < bpp) {               // Avg / Paeth: serial in x, one lane per byte position mod bpp
      int a = 0, cc = 0;
      if (ft == 3) {
#pragma unroll 4
        for (int i = lane; i < rb; i += bpp) {
          const int b = prev ? prev[i] : 0;
          a = (uint8_t)(cur[i] + ((a + b) >> 1));
          cur[i] = (uint8_t)a;
        }
      } else {
#pragma unroll 4
        for (int i = lane; i < rb; i += bpp) {
          const int b = prev ? prev[i] : 0;
          a = (uint8_t)(cur[i] + paeth(a, b, cc));
          cur[i] = (uint8_t)a;
          cc = b;
        }
      }
    }
    __syncwarp();
    uint8_t* o = out + (int64_t)3 * y * W;
    for (int x = lane; x < W; x += 32) {
      uint32_t r, g, b;
      if (depth < 8) {                                // grey or palette, 1 / 2 / 4 bits, first pixel in the high bits
        const int per = 8 / depth;
        const uint32_t v = (cur[x / per] >> (8 - depth * (x % per + 1))) & ((1u << depth) - 1);
        if (ct == 3) { r = pal[warp][3 * v]; g = pal[warp][3 * v + 1]; b = pal[warp][3 * v + 2]; }
        else { r = g = b = v * (depth == 1 ? 255u : depth == 2 ? 85u : 17u); }
      } else if (depth == 8) {
        const uint8_t* p = cur + (int64_t)x * bpp;
        if (ct == 0 || ct == 4) { r = g = b = p[0]; }
        else if (ct == 3) { r = pal[warp][3 * p[0]]; g = pal[warp][3 * p[0] + 1]; b = pal[warp][3 * p[0] + 2]; }
        else { r = p[0]; g = p[1]; b = p[2]; }
      } else {                                        // 16 bits, big-endian samples
        const uint8_t* p = cur + (int64_t)x * bpp;
        if (ct == 0) { r = g = b = p[0] ? 255u : p[1]; }          // I;16 -> RGB saturates
        else if (ct == 4) { r = g = b = p[0]; }                   // high byte
        else { r = p[0]; g = p[2]; b = p[4]; }
      }
      o[3 * x] = (uint8_t)r; o[3 * x + 1] = (uint8_t)g; o[3 * x + 2] = (uint8_t)b;
    }
  }
}

}  // namespace png
}  // namespace gnc

using namespace gnc;

extern "C" {

int gnc_png_pack(const uint8_t* const* datas, const int64_t* sizes, int n, int threads, uint8_t* stream_out,
                 int64_t stream_capacity, gnc_png_image_t* images_out, int32_t* index_out, int64_t* totals) {
  GNC_REQUIRE(n >= 0 && (n == 0 || (datas && sizes && stream_out && images_out && index_out)) && totals, "png_pack: bad arguments");
  std::vector<std::vector<png::Segment>> segs((size_t)n);
  std::vector<gnc_png_image_t> parsed((size_t)n);
  std::vector<int> ok((size_t)n, 0);
  const int nt = threads < 1 ? 1 : (threads > 32 ? 32 : threads);
  auto parallel = [&](int count, auto&& fn) {
    if (nt == 1 || count < 8) { for (int i = 0; i < count; ++i) fn(i); return; }
    std::vector<std::thread> pool;
    for (int t = 0; t < nt; ++t) pool.emplace_back([&, t]() { for (int i = t; i < count; i += nt) fn(i); });
    for (auto& th : pool) th.join();
  };
  parallel(n, [&](int i) { ok[i] = png::parse(datas[i], sizes[i], &parsed[i], segs[i]) == GNC_OK; });
  std::vector<int> order;
  for (int i = 0; i < n; ++i)
    if (ok[i]) order.push_back(i);
  // longest stream first: a batch takes at least as long as its longest serial stream
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return parsed[a].stream_bytes > parsed[b].stream_bytes; });
  const int m = (int)order.size();
  int64_t off = 0, raw = 0, pixels = 0;
  for (int j = 0; j < m; ++j) {
    gnc_png_image_t& d = images_out[j];
    d = parsed[order[j]];
    d.stream_offset = off; d.raw_offset = raw; d.pixel_offset = pixels;
    index_out[j] = order[j];
    off += d.stream_bytes; raw += d.raw_bytes; pixels += (int64_t)d.width * d.height;
  }
  GNC_REQUIRE(off <= stream_capacity, "png_pack: stream buffer too small");
  parallel(m, [&](int j) {
    uint8_t* dst = stream_out + images_out[j].stream_offset;
    const uint8_t* src = datas[order[j]];
    for (const png::Segment& s : segs[order[j]]) { memcpy(dst, src + s.offset, (size_t)s.bytes); dst += s.bytes; }
  });
  totals[0] = m; totals[1] = off; totals[2] = raw; totals[3] = pixels;
  return GNC_OK;
}

int gnc_png_decode_rgb_u8(const uint8_t* stream, const gnc_png_image_t* images, int B, uint8_t* raw, uint8_t* out,
                          int32_t* status, gnc_stream_t stream_) {
  GNC_REQUIRE(B >= 0, "png_decode: bad sizes");
  if (B == 0) return GNC_OK;
  GNC_REQUIRE(stream && images && raw && out && status, "png_decode: null pointer");
  cudaStream_t st = (cudaStream_t)stream_;
  png::png_inflate_kernel<<<(unsigned)B, 32, 0, st>>>(stream, images, B, raw, status);
  if (int rc = check_launch("png_inflate_kernel")) return rc;
  png::png_unfilter_kernel<<<(unsigned)ceil_div<int>(B, png::kWarps), 32 * png::kWarps, 0, st>>>(images, B, raw, out, status);
  return check_launch("png_unfilter_kernel");
}

}  // extern "C"
