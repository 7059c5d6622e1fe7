// Baseline JPEG decode on the device: the other half of the reference's input staging,
//   Image.open(path).convert('RGB')       utils/dataloader.py:34 (ImageFolder's loader),
//                                         utils/image_to_graph/image_to_graph_optimized.py:65-68, utils/inference.py:47
// i.e. libjpeg(-turbo) behind Pillow with its defaults: Huffman sequential DCT, the accurate integer inverse DCT
// (JDCT_ISLOW, jidctint.c), "fancy" triangle-filter chroma upsampling (jdsample.c) and the 16-bit fixed-point
// YCbCr -> RGB tables (jdcolor.c).  libjpeg is an un-vendored dependency of an un-vendored dependency (Pillow); its
// decoder is a published integer algorithm, restated here stage by stage so that the pixels are bit for bit the ones
// Pillow hands the reference (tests/test_gpu_jpeg.py compares with Pillow on generated files and on the reference's
// shipped JPEGs).
//
// Scope: what `Image.save(..., 'JPEG')` and ordinary cameras write and the shipped dataset uses - 8-bit baseline /
// extended-sequential Huffman (SOF0 / SOF1), one interleaved scan, greyscale or YCbCr with 4:4:4, 4:2:2 (h2v1) or 4:2:0
// (h2v2) chroma, optional restart intervals, optional JFIF / EXIF / ICC segments (skipped; Pillow's convert('RGB') does
// not apply them either).  Progressive files (SOF2, 8-bit Huffman) with the same frame layouts are decoded by a second
// entry point, on request (utils/jpeg.decode_batch(..., progressive=True)).  Anything else (arithmetic coding, CMYK /
// Adobe transforms, 12-bit, multi-scan sequential, and progressive files libjpeg would not decode by the plain path -
// see parse_progressive) is reported as unsupported and decoded by Pillow on the host (utils/staging.py) - same pixels
// either way.
//
// Stages:
//   host   gnc_jpeg_parse         : markers -> geometry, dequantisation tables (natural order), Huffman decode tables
//                                   (9-bit lookahead + canonical maxcode / valptr for longer codes), scan position
//   device jpeg_huffman_kernel    : one warp per image.  Entropy decode is sequential by nature (no restart markers in
//                                   Pillow's files), but Huffman streams are self-synchronising: the warp's 32 lanes decode
//                                   32 segments of the scan from guessed states and iterate until every segment starts where
//                                   its predecessor stopped (see "parallel form" below); short scans and scans with restart
//                                   intervals are walked by one thread (64-bit bit buffer, byte unstuffing)
//          jpeg_idct_kernel       : one thread per 8 x 8 block, jidctint.c's two passes in registers, range-limited
//                                   samples into per-component planes
//          jpeg_color_kernel      : one thread per output pixel: fancy upsampling of the chroma planes evaluated at the
//                                   pixel (libjpeg's rounding terms and edge rules) + the fixed-point colour tables
// Progressive files:
//   host   gnc_jpeg_pack_progressive : markers -> frame descriptor (quantisation tables latched at each component's first
//                                   scan), one record per scan with the Huffman tables and restart interval in force
//                                   at that scan, and the partition of the scans into chains (scans linked by a common
//                                   coefficient of a common component), longest first across the batch
//   device jpeg_progressive_kernel : one lane per chain walks its scans in file order with jdphuff.c's four procedures
//                                   (DC first / refine, AC first / refine) into the zeroed coefficient buffer; the same
//                                   jpeg_idct_kernel and jpeg_color_kernel then run on the frame descriptors
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <thread>
#include <vector>

#include "common.cuh"

namespace gnc {
namespace jpeg {

constexpr int kLook = 9;                      // lookahead bits of the Huffman tables

// zigzag position -> natural (row-major) position
__constant__ uint8_t c_natural[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                      41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                      30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
static const uint8_t h_natural[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                      41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                      30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

// ---- entropy decode -------------------------------------------------------------------------------------------------
// A single thread runs at a few hundred MIPS on this machine (every instruction waits ~5 cycles for the one before it),
// so the loop is written for a short dependent chain per symbol: ONE refill check per symbol (>= 32 valid bits cover the
// longest code + the longest value), the code and its value bits taken from the same 32-bit window, the tables of the
// warp's image in shared memory, four stream bytes appended at a time unless one of them is 0xFF.
struct BitReader {
  const uint8_t* p;        // next byte of the stream
  const uint8_t* end;
  uint64_t acc;            // bits, MSB-aligned
  int n;                   // valid bits in acc
  bool marker;             // a marker (FF xx, xx != 0) was met: feed zeros, as libjpeg does past the end of a segment
};

__device__ __forceinline__ void refill_bytes(BitReader& br) {
  while (br.n <= 56) {
    uint32_t byte = 0;
    if (!br.marker && br.p < br.end) {
      byte = *br.p;
      if (byte == 0xFF) {
        const uint32_t nxt = (br.p + 1 < br.end) ? br.p[1] : 0xD9;
        if (nxt == 0) br.p += 2;                 // stuffed zero: a data byte FF
        else { br.marker = true; byte = 0; }     // stay on the marker
      } else {
        br.p += 1;
      }
    }
    br.acc |= (uint64_t)byte << (56 - br.n);
    br.n += 8;
  }
}
// at least 32 valid bits
__device__ __forceinline__ void ensure32(BitReader& br) {
  if (br.n >= 32) return;
  if (!br.marker && br.p + 4 <= br.end) {
    const uint32_t b0 = br.p[0], b1 = br.p[1], b2 = br.p[2], b3 = br.p[3];      // independent loads
    if (b0 != 0xFF && b1 != 0xFF && b2 != 0xFF && b3 != 0xFF) {
      const uint32_t w = (b0 << 24) | (b1 << 16) | (b2 << 8) | b3;
      br.acc |= (uint64_t)w << (32 - br.n);
      br.n += 32;
      br.p += 4;
      return;
    }
  }
  refill_bytes(br);
}
// one Huffman symbol and the `size` value bits behind it (jdhuff.c: lookahead table, canonical code walk, HUFF_EXTEND);
// for AC symbols size = low nibble, for DC symbols size = the symbol.  Returns the symbol, the extended value in `val`.
template <bool kDC>
__device__ __forceinline__ int decode_pair(BitReader& br, const gnc_jpeg_huff_t* t, int& val) {
  ensure32(br);
  const uint32_t w = (uint32_t)(br.acc >> 32);
  const uint32_t look = t->look[w >> (32 - kLook)];
  int len, sym;
  if (look) {
    len = (int)(look >> 8); sym = (int)(look & 0xff);
  } else {
    len = kLook + 1;
    int32_t code = (int32_t)(w >> (32 - len));
    while (len <= 16 && code > t->maxcode[len]) { ++len; code = (int32_t)(w >> (32 - len)); }
    if (len > 16) { len = 16; sym = 0; }         // corrupt stream: libjpeg warns and uses 0
    else sym = t->vals[(code + t->valoff[len]) & 0xff];
  }
  const int s = kDC ? (sym & 15) : (sym & 15);
  const uint32_t bits = s ? ((w << len) >> (32 - s)) : 0u;                      // len + s <= 27
  val = s ? ((int)bits < (1 << (s - 1)) ? (int)bits - (1 << s) + 1 : (int)bits) : 0;
  br.acc <<= (len + s);
  br.n -= (len + s);
  return sym;
}

constexpr int kHuffWarps = 4;

// sequential form: one thread walks the whole scan (images with restart intervals, very short scans, and the reference
// the parallel form below is tested against)
__device__ __noinline__ void decode_sequential(const uint8_t* __restrict__ stream, const gnc_jpeg_image_t* im,
                                               const gnc_jpeg_huff_t* tabs, int16_t* __restrict__ coef) {
  BitReader br;
  br.p = stream + im->scan_offset;
  br.end = br.p + im->scan_bytes;
  br.acc = 0; br.n = 0; br.marker = false;
  int16_t* cimg = coef + im->coef_offset;
  const int ncomp = im->ncomp, mcu_x = im->mcu_x, mcu_y = im->mcu_y;
  const int h0 = im->hsamp[0], v0 = im->vsamp[0];
  const int64_t base1 = (int64_t)mcu_x * h0 * mcu_y * v0 * 64;          // chroma planes: one block per MCU each
  const int64_t base2 = base1 + (int64_t)mcu_x * mcu_y * 64;
  const gnc_jpeg_huff_t* dc0 = tabs + im->dc_tab[0];
  const gnc_jpeg_huff_t* ac0 = tabs + 4 + im->ac_tab[0];
  const gnc_jpeg_huff_t* dc1 = tabs + im->dc_tab[ncomp > 1 ? 1 : 0];
  const gnc_jpeg_huff_t* ac1 = tabs + 4 + im->ac_tab[ncomp > 1 ? 1 : 0];
  const gnc_jpeg_huff_t* dc2 = tabs + im->dc_tab[ncomp > 2 ? 2 : 0];
  const gnc_jpeg_huff_t* ac2 = tabs + 4 + im->ac_tab[ncomp > 2 ? 2 : 0];
  int pred0 = 0, pred1 = 0, pred2 = 0;
  auto block = [&](int16_t* blk, const gnc_jpeg_huff_t* dct, const gnc_jpeg_huff_t* act, int& pred) {
    int v;
    decode_pair<true>(br, dct, v);
    pred += v;
    blk[0] = (int16_t)pred;
    int k = 1;
    while (k < 64) {
      const int sym = decode_pair<false>(br, act, v);
      const int r = sym >> 4;
      if (sym & 15) {
        k += r;
        blk[c_natural[k & 63]] = (int16_t)v;
        ++k;
      } else {
        if (r != 15) break;                      // end of block
        k += 16;                                 // sixteen zeros
      }
    }
  };
  const int restart = im->restart_interval;
  int to_restart = restart;
  for (int my = 0; my < mcu_y; ++my) {
    for (int mx = 0; mx < mcu_x; ++mx) {
      if (restart && to_restart == 0) {
        // byte-align, step over the RSTn marker, reset the predictions (jdhuff.c process_restart)
        br.acc = 0; br.n = 0;
        if (br.marker) { br.p += 2; br.marker = false; }
        else {                                   // the marker has not been reached by the reader yet: find it
          while (br.p + 1 < br.end && !(br.p[0] == 0xFF && br.p[1] >= 0xD0 && br.p[1] <= 0xD7)) ++br.p;
          br.p += 2;
        }
        pred0 = pred1 = pred2 = 0;
        to_restart = restart;
      }
      for (int by = 0; by < v0; ++by)
        for (int bx = 0; bx < h0; ++bx)
          block(cimg + ((int64_t)(my * v0 + by) * (mcu_x * h0) + (mx * h0 + bx)) * 64, dc0, ac0, pred0);
      if (ncomp == 3) {
        block(cimg + base1 + ((int64_t)my * mcu_x + mx) * 64, dc1, ac1, pred1);
        block(cimg + base2 + ((int64_t)my * mcu_x + mx) * 64, dc2, ac2, pred2);
      }
      if (restart) --to_restart;
    }
  }
}

// ---- parallel form: the 32 lanes of the image's warp decode 32 segments of its scan ---------------------------------------
// Huffman streams are self-synchronising: a decoder started at an arbitrary bit soon falls into step with the true one.
// (Weissenberger & Schmidt, "Massively Parallel Huffman Decoding on GPUs", ICPP 2018; for JPEG the state that has to agree
// is the bit position, the block's position in the MCU - it selects the tables - and the coefficient index.)
//   0. the warp removes the stuffed zeros (FF 00 -> FF) into a scratch copy of the scan: a position is then a plain bit
//      index and a 32-bit window two aligned loads and a funnel shift - no refill state to hand from lane to lane;
//   1. lane i decodes segment i from a guessed state (start of an MCU) up to the segment's end and records the state it
//      leaves in and the number of blocks it completed;
//   2. lane i > 0 compares its entry state with the exit state of lane i - 1 and decodes again from there if they differ;
//      repeated until no entry changes.  Lane 0 starts from the true state, so at the fixed point every entry is true
//      (at worst after 31 rounds, in practice after one or two);
//   3. prefix sum of the block counts -> the first block of every segment; 4. the lanes decode once more and write the
//      coefficients (DC still as differences); 5. per component a warp scan turns the DC differences into DC values.
struct SegState { uint32_t T; int z, k; };
__device__ __forceinline__ bool same(const SegState& a, const SegState& b) { return a.T == b.T && a.z == b.z && a.k == b.k; }
__device__ __forceinline__ uint32_t window32(const uint8_t* us, uint32_t T) {
  const uint32_t idx = T >> 3;
  const uint32_t* wp = reinterpret_cast<const uint32_t*>(us + (idx & ~3u));
  const uint32_t hi = __byte_perm(wp[0], 0, 0x0123), lo = __byte_perm(wp[1], 0, 0x0123);
  return __funnelshift_l(lo, hi, (idx & 3u) * 8u + (T & 7u));
}
// one symbol + its value bits at bit T of the unstuffed stream (same tables and rules as decode_pair)
__device__ __forceinline__ int symbol_at(const uint8_t* us, uint32_t& T, const gnc_jpeg_huff_t* t, int& val) {
  const uint32_t w = window32(us, T);
  const uint32_t look = t->look[w >> (32 - kLook)];
  int len, sym;
  if (look) {
    len = (int)(look >> 8); sym = (int)(look & 0xff);
  } else {
    len = kLook + 1;
    int32_t code = (int32_t)(w >> (32 - len));
    while (len <= 16 && code > t->maxcode[len]) { ++len; code = (int32_t)(w >> (32 - len)); }
    if (len > 16) { len = 16; sym = 0; }
    else sym = t->vals[(code + t->valoff[len]) & 0xff];
  }
  const int s = sym & 15;
  const uint32_t bits = s ? ((w << len) >> (32 - s)) : 0u;
  val = s ? ((int)bits < (1 << (s - 1)) ? (int)bits - (1 << s) + 1 : (int)bits) : 0;
  T += (uint32_t)(len + s);
  return sym;
}

struct ImgGeom {
  int16_t* cimg;
  int mcu_x, h0, nY, bpm;                         // luma blocks per MCU, blocks per MCU
  int64_t base1, base2, n_blocks;
  const gnc_jpeg_huff_t *dcY, *acY, *dc1, *ac1, *dc2, *ac2;
};
__device__ __forceinline__ int16_t* block_ptr(const ImgGeom& g, int64_t blk) {
  const int64_t mcu = blk / g.bpm;
  const int z = (int)(blk - mcu * g.bpm);
  const int my = (int)(mcu / g.mcu_x), mx = (int)(mcu - (int64_t)my * g.mcu_x);
  if (z < g.nY) {
    const int by = z / g.h0, bx = z - by * g.h0;
    const int v0 = g.nY / g.h0;
    return g.cimg + ((int64_t)(my * v0 + by) * (g.mcu_x * g.h0) + (mx * g.h0 + bx)) * 64;
  }
  return g.cimg + (z == g.nY ? g.base1 : g.base2) + mcu * 64;
}
// decode from `st` until the position reaches t_end; kWrite: coefficients go to the blocks starting at `blk`.
// The 32 lanes of a warp run this loop on 32 different segments, so the symbol step is written without branches on the
// kind of symbol (DC / coefficient / zero run / end of block take the same instructions, selected by predicates) and the
// block bookkeeping at the end of a block - some lane ends a block in almost every iteration - has no divisions: the
// block's place is carried as (MCU row, MCU column, index in the MCU).
template <bool kWrite>
__device__ __forceinline__ void run_segment(const uint8_t* us, const ImgGeom& g, SegState& st, uint32_t t_end, int& nblocks, int64_t blk) {
  nblocks = 0;
  uint32_t T = st.T;
  int z = st.z, k = st.k;
  int mx = 0, my = 0;
  int16_t* bp = nullptr;
  const int hsh = g.h0 - 1;                         // h0 is 1 or 2: z -> (z >> hsh, z & hsh) inside the MCU
  const int v0 = g.nY / g.h0;
  auto place = [&]() -> int16_t* {
    if (z < g.nY) return g.cimg + ((int64_t)(my * v0 + (z >> hsh)) * (g.mcu_x * g.h0) + (mx * g.h0 + (z & hsh))) * 64;
    return g.cimg + (z == g.nY ? g.base1 : g.base2) + ((int64_t)my * g.mcu_x + mx) * 64;
  };
  int64_t left = 0;                                 // blocks that may still be written
  if (kWrite) {
    const int64_t mcu = blk / g.bpm;
    my = (int)(mcu / g.mcu_x); mx = (int)(mcu - (int64_t)my * g.mcu_x);
    left = g.n_blocks - blk;
    bp = left > 0 ? place() : nullptr;
  }
  const gnc_jpeg_huff_t* dct = z < g.nY ? g.dcY : (z == g.nY ? g.dc1 : g.dc2);
  const gnc_jpeg_huff_t* act = z < g.nY ? g.acY : (z == g.nY ? g.ac1 : g.ac2);
  while (T < t_end) {
    const bool isdc = k == 0;
    int v;
    const int sym = symbol_at(us, T, isdc ? dct : act, v);
    const int s = sym & 15, r = isdc ? 0 : sym >> 4;
    const bool coef = isdc || s != 0;
    const int kp = isdc ? 0 : k + r;
    if (kWrite && coef && bp && kp < 64) bp[c_natural[kp]] = (int16_t)v;       // DC: the DIFFERENCE; step 5 integrates
    k = coef ? kp + 1 : (r == 15 ? k + 16 : 64);
    if (k >= 64) {                                  // end of block
      k = 0;
      ++nblocks;
      ++z;
      if (z == g.bpm) { z = 0; if (kWrite) { ++mx; if (mx == g.mcu_x) { mx = 0; ++my; } } }
      dct = z < g.nY ? g.dcY : (z == g.nY ? g.dc1 : g.dc2);
      act = z < g.nY ? g.acY : (z == g.nY ? g.ac1 : g.ac2);
      if (kWrite) { --left; bp = left > 0 ? place() : nullptr; }
    }
  }
  st.T = T; st.z = z; st.k = k;
}

constexpr int kMinParallelBytes = 4096;           // shorter scans: one thread is as fast

__global__ void __launch_bounds__(32 * kHuffWarps) jpeg_huffman_kernel(const uint8_t* __restrict__ stream,
                                                                       const gnc_jpeg_image_t* __restrict__ infos, int B,
                                                                       int16_t* __restrict__ coef, uint8_t* __restrict__ scratch,
                                                                       int force_sequential) {
  extern __shared__ __align__(16) uint8_t s_tables[];                   // [kHuffWarps][8] gnc_jpeg_huff_t
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int img = blockIdx.x * kHuffWarps + warp;
  if (img >= B) return;
  const gnc_jpeg_image_t* im = infos + img;
  gnc_jpeg_huff_t* tabs = reinterpret_cast<gnc_jpeg_huff_t*>(s_tables) + warp * 8;
  {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(im->huff);
    uint32_t* dst = reinterpret_cast<uint32_t*>(tabs);
    for (int i = lane; i < (int)(8 * sizeof(gnc_jpeg_huff_t) / 4); i += 32) dst[i] = __ldg(src + i);
  }
  __syncwarp();
  if (!scratch || (force_sequential & 1) || im->restart_interval || im->scan_bytes < kMinParallelBytes) {
    if (lane == 0) decode_sequential(stream, im, tabs, coef);
    return;
  }
  const unsigned kFull = 0xffffffffu;
  // 0. unstuffed copy of the scan
  const uint8_t* raw = stream + im->scan_offset;
  const uint32_t nraw = (uint32_t)im->scan_bytes;
  uint8_t* us = scratch + (((uint64_t)im->scan_offset + 3u) & ~(uint64_t)3u) + 16ull * (uint64_t)img;
  uint32_t outpos = 0, carry = 0;
  for (uint32_t base = 0; base < nraw; base += 128) {                   // 4 bytes per lane: a byte is dropped iff it is
    const uint32_t i0 = base + 4u * lane;                               // the 00 behind an FF
    uint32_t by[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) by[j] = i0 + j < nraw ? raw[i0 + j] : 0x100u;
    uint32_t prev = __shfl_up_sync(kFull, by[3], 1);
    if (lane == 0) prev = carry;
    bool keep[4];
    int nk = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      keep[j] = by[j] < 0x100u && !(by[j] == 0u && prev == 0xFFu);
      nk += keep[j] ? 1 : 0;
      prev = by[j];
    }
    int incl = nk;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(kFull, incl, o); if (lane >= o) incl += t; }
    uint8_t* dst = us + outpos + (incl - nk);
    int at = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (keep[j]) dst[at] = (uint8_t)by[j];
      at += keep[j] ? 1 : 0;
    }
    outpos += __shfl_sync(kFull, incl, 31);
    carry = __shfl_sync(kFull, by[3], 31);
  }
  if (lane < 12) us[outpos + lane] = 0;           // zeros behind the data: a window may read past the last byte
  __syncwarp();
  const uint32_t total_bits = outpos * 8u;
  ImgGeom g;
  g.cimg = coef + im->coef_offset;
  g.mcu_x = im->mcu_x; g.h0 = im->hsamp[0]; g.nY = im->hsamp[0] * im->vsamp[0];
  g.bpm = g.nY + (im->ncomp == 3 ? 2 : 0);
  g.base1 = (int64_t)im->mcu_x * im->mcu_y * g.nY * 64;
  g.base2 = g.base1 + (int64_t)im->mcu_x * im->mcu_y * 64;
  g.n_blocks = im->n_blocks;
  g.dcY = tabs + im->dc_tab[0]; g.acY = tabs + 4 + im->ac_tab[0];
  g.dc1 = tabs + im->dc_tab[im->ncomp > 1 ? 1 : 0]; g.ac1 = tabs + 4 + im->ac_tab[im->ncomp > 1 ? 1 : 0];
  g.dc2 = tabs + im->dc_tab[im->ncomp > 2 ? 2 : 0]; g.ac2 = tabs + 4 + im->ac_tab[im->ncomp > 2 ? 2 : 0];
  // 1. speculative pass
  const uint32_t seg = ((total_bits + 31u) / 32u + 7u) & ~7u;            // bits per segment
  const uint32_t t_end = min(total_bits, (uint32_t)(lane + 1) * seg);
  SegState entry;
  entry.T = min(total_bits, (uint32_t)lane * seg); entry.z = 0; entry.k = 0;
  SegState ex = entry;
  int nblk;
  run_segment<false>(us, g, ex, t_end, nblk, 0);
  // 2. until every lane starts where its predecessor stopped
  int rounds = 0, reruns = 0;
  for (int round = 0; round < 32; ++round) {
    SegState pe;
    pe.T = __shfl_up_sync(kFull, ex.T, 1); pe.z = __shfl_up_sync(kFull, ex.z, 1); pe.k = __shfl_up_sync(kFull, ex.k, 1);
    const bool need = lane > 0 && !same(pe, entry);
    if (!__any_sync(kFull, need)) break;
    ++rounds;
    if (need) {
      ++reruns;
      entry = pe;
      ex = pe;
      run_segment<false>(us, g, ex, t_end, nblk, 0);
    }
  }
  if ((force_sequential & 2) && img < 3) {
    const unsigned long long t1 = clock64();
    printf("img %d lane %2d: rounds %d reruns %d entry (T %u z %d k %d) blocks %d seg %u bits\n", img, lane, rounds, reruns, entry.T,
           entry.z, entry.k, nblk, seg);
    (void)t1;
  }
  // 3. first block of every segment
  int incl = nblk;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(kFull, incl, o); if (lane >= o) incl += v; }
  // 4. write pass
  {
    SegState st = entry;
    int n2;
    run_segment<true>(us, g, st, t_end, n2, (int64_t)(incl - nblk));
  }
  __syncwarp();
  // 5. DC differences -> DC values, per component in decode order
  const int64_t nmcu = (int64_t)im->mcu_x * im->mcu_y;
  for (int c = 0; c < im->ncomp; ++c) {
    const int64_t len = c == 0 ? nmcu * g.nY : nmcu;
    const int64_t per = (len + 31) / 32, lo = min(len, per * lane), hi = min(len, lo + per);
    auto ptr = [&](int64_t j) -> int16_t* {
      if (c == 0) { const int64_t mcu = j / g.nY; return block_ptr(g, mcu * g.bpm + (j - mcu * g.nY)); }
      return g.cimg + (c == 1 ? g.base1 : g.base2) + j * 64;
    };
    int sum = 0;
    for (int64_t j = lo; j < hi; ++j) sum += ptr(j)[0];
    int run = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(kFull, run, o); if (lane >= o) run += v; }
    int acc = run - sum;
    for (int64_t j = lo; j < hi; ++j) { int16_t* q = ptr(j); acc += q[0]; q[0] = (int16_t)acc; }
  }
}

// ---- inverse DCT (jidctint.c, jpeg_idct_islow) -------------------------------------------------------------------------
constexpr int CONST_BITS = 13, PASS1_BITS = 2;
constexpr int FIX_0_298631336 = 2446, FIX_0_390180644 = 3196, FIX_0_541196100 = 4433, FIX_0_765366865 = 6270,
              FIX_0_899976223 = 7373, FIX_1_175875602 = 9633, FIX_1_501321110 = 12299, FIX_1_847759065 = 15137,
              FIX_1_961570560 = 16069, FIX_2_053119869 = 16819, FIX_2_562915447 = 20995, FIX_3_072711026 = 25172;

__device__ __forceinline__ int descale(int x, int n) { return (x + (1 << (n - 1))) >> n; }
// IDCT_range_limit[x & RANGE_MASK]: x + 128 clamped to 0..255 for |x| < 512 (and libjpeg's wrap-around beyond)
__device__ __forceinline__ uint8_t range_limit(int x) {
  const int v = x & 1023;
  return (uint8_t)(v < 128 ? v + 128 : (v < 512 ? 255 : (v < 896 ? 0 : v - 896)));
}

__device__ __forceinline__ void idct_1d(const int in[8], int out[8], bool pass1) {
  int z2 = in[2], z3 = in[6];
  int z1 = (z2 + z3) * FIX_0_541196100;
  int tmp2 = z1 + z3 * (-FIX_1_847759065);
  int tmp3 = z1 + z2 * FIX_0_765366865;
  z2 = in[0]; z3 = in[4];
  int tmp0 = (z2 + z3) << CONST_BITS;
  int tmp1 = (z2 - z3) << CONST_BITS;
  const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
  tmp0 = in[7]; tmp1 = in[5]; tmp2 = in[3]; tmp3 = in[1];
  z1 = tmp0 + tmp3; z2 = tmp1 + tmp2; z3 = tmp0 + tmp2;
  int z4 = tmp1 + tmp3;
  const int z5 = (z3 + z4) * FIX_1_175875602;
  tmp0 *= FIX_0_298631336; tmp1 *= FIX_2_053119869; tmp2 *= FIX_3_072711026; tmp3 *= FIX_1_501321110;
  z1 *= -FIX_0_899976223; z2 *= -FIX_2_562915447; z3 *= -FIX_1_961570560; z4 *= -FIX_0_390180644;
  z3 += z5; z4 += z5;
  tmp0 += z1 + z3; tmp1 += z2 + z4; tmp2 += z2 + z3; tmp3 += z1 + z4;
  const int sh = pass1 ? CONST_BITS - PASS1_BITS : CONST_BITS + PASS1_BITS + 3;
  out[0] = descale(tmp10 + tmp3, sh); out[7] = descale(tmp10 - tmp3, sh);
  out[1] = descale(tmp11 + tmp2, sh); out[6] = descale(tmp11 - tmp2, sh);
  out[2] = descale(tmp12 + tmp1, sh); out[5] = descale(tmp12 - tmp1, sh);
  out[3] = descale(tmp13 + tmp0, sh); out[4] = descale(tmp13 - tmp0, sh);
}

// one thread per block; blocks of all images and components are numbered through `block_offset`
__global__ void __launch_bounds__(128) jpeg_idct_kernel(const gnc_jpeg_image_t* __restrict__ infos, int B, const int16_t* __restrict__ coef,
                                                        uint8_t* __restrict__ planes, int64_t total_blocks) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total_blocks) return;
  // image of this block: binary search over the per-image block offsets
  int lo = 0, hi = B - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (infos[mid].block_offset <= g) lo = mid; else hi = mid - 1;
  }
  const gnc_jpeg_image_t* im = infos + lo;
  int64_t rel = g - im->block_offset;
  int c = 0;
  int bwc = 0;
  for (; c < im->ncomp; ++c) {
    bwc = im->mcu_x * im->hsamp[c];
    const int64_t nb = (int64_t)bwc * im->mcu_y * im->vsamp[c];
    if (rel < nb) break;
    rel -= nb;
  }
  const int by = (int)(rel / bwc), bx = (int)(rel - (int64_t)by * bwc);
  const int16_t* blk = coef + im->coef_offset + (g - im->block_offset) * 64;
  const uint16_t* q = im->quant[im->qtab[c]];
  int ws[64];
#pragma unroll
  for (int col = 0; col < 8; ++col) {                     // pass 1: columns, dequantised
    int in[8], out[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) in[r] = (int)blk[r * 8 + col] * (int)q[r * 8 + col];
    idct_1d(in, out, true);
#pragma unroll
    for (int r = 0; r < 8; ++r) ws[r * 8 + col] = out[r];
  }
  // component plane: MCU-padded width bwc * 8
  int64_t plane_off = im->plane_offset;
  for (int cc = 0; cc < c; ++cc) plane_off += (int64_t)im->mcu_x * im->hsamp[cc] * 8 * im->mcu_y * im->vsamp[cc] * 8;
  uint8_t* dst = planes + plane_off + ((int64_t)by * 8) * (bwc * 8) + bx * 8;
#pragma unroll
  for (int r = 0; r < 8; ++r) {                           // pass 2: rows
    int in[8], out[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) in[k] = ws[r * 8 + k];
    idct_1d(in, out, false);
    uint32_t w0 = 0, w1 = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) { w0 |= (uint32_t)range_limit(out[k]) << (8 * k); w1 |= (uint32_t)range_limit(out[4 + k]) << (8 * k); }
    *reinterpret_cast<uint2*>(dst + (int64_t)r * (bwc * 8)) = make_uint2(w0, w1);
  }
}

// ---- chroma upsampling + colour conversion, evaluated per output pixel ---------------------------------------------------
// jdsample.c: the upsampled value at an output position is a fixed function of at most 4 samples of the component:
//   h2v1 fancy: out[2i] = (3 s[i] + s[i-1] + 1) >> 2, out[2i+1] = (3 s[i] + s[i+1] + 2) >> 2, edges copy s[0] / s[last]
//   h2v2 fancy: vertically v(i) = 3 s[near][i] + s[far][i] (near = the sample row, far = the row above for the upper
//               output row and below for the lower one; the first / last REAL rows stand in for rows beyond the image),
//               then out[2i] = (3 v(i) + v(i-1) + 8) >> 4, out[2i+1] = (3 v(i) + v(i+1) + 7) >> 4,
//               edges (4 v(0) + 8) >> 4 and (4 v(last) + 7) >> 4
// with `last` = the component's true downsampled width - 1 (not the MCU padding).  Components of at most 2 samples in a
// row are replicated instead (jinit_upsampler).
__device__ __forceinline__ int upsampled(const uint8_t* plane, int pw, int dw, int dh, int hfac, int vfac, int x, int y) {
  if (hfac == 1 && vfac == 1) return plane[(int64_t)y * pw + x];
  const int i = x >> 1;
  if (vfac == 1) {                                        // h2v1
    const uint8_t* row = plane + (int64_t)y * pw;
    if (dw <= 2) return row[i];
    const int s = row[i];
    if ((x & 1) == 0) return i == 0 ? s : (3 * s + row[i - 1] + 1) >> 2;
    return i == dw - 1 ? s : (3 * s + row[i + 1] + 2) >> 2;
  }
  const int j = y >> 1;                                   // h2v2
  if (dw <= 2) return plane[(int64_t)j * pw + i];
  int jf = (y & 1) ? j + 1 : j - 1;
  jf = jf < 0 ? 0 : (jf > dh - 1 ? dh - 1 : jf);
  const uint8_t* near = plane + (int64_t)j * pw;
  const uint8_t* far = plane + (int64_t)jf * pw;
  const int v = 3 * near[i] + far[i];
  if ((x & 1) == 0) {
    if (i == 0) return (4 * v + 8) >> 4;
    return (3 * v + (3 * near[i - 1] + far[i - 1]) + 8) >> 4;
  }
  if (i == dw - 1) return (4 * v + 7) >> 4;
  return (3 * v + (3 * near[i + 1] + far[i + 1]) + 7) >> 4;
}
__device__ __forceinline__ uint8_t clamp255(int v) { return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v)); }

__global__ void __launch_bounds__(256) jpeg_color_kernel(const gnc_jpeg_image_t* __restrict__ infos, int B, const uint8_t* __restrict__ planes,
                                                         uint8_t* __restrict__ out, int64_t total_pixels) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total_pixels) return;
  int lo = 0, hi = B - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (infos[mid].pixel_offset <= g) lo = mid; else hi = mid - 1;
  }
  const gnc_jpeg_image_t* im = infos + lo;
  const int64_t rel = g - im->pixel_offset;
  const int y = (int)(rel / im->width), x = (int)(rel - (int64_t)y * im->width);
  const uint8_t* p0 = planes + im->plane_offset;
  const int pw0 = im->mcu_x * im->hsamp[0] * 8;
  const int Y = p0[(int64_t)y * pw0 + x];
  uint8_t* o = out + (im->pixel_offset + rel) * 3;
  if (im->ncomp == 1) { o[0] = o[1] = o[2] = (uint8_t)Y; return; }
  const int64_t n0 = (int64_t)pw0 * im->mcu_y * im->vsamp[0] * 8;
  const int pw1 = im->mcu_x * im->hsamp[1] * 8;
  const int64_t n1 = (int64_t)pw1 * im->mcu_y * im->vsamp[1] * 8;
  const int hf = im->hsamp[0] / im->hsamp[1], vf = im->vsamp[0] / im->vsamp[1];
  const int dw = (im->width * im->hsamp[1] + im->hsamp[0] - 1) / im->hsamp[0];       // true downsampled size
  const int dh = (im->height * im->vsamp[1] + im->vsamp[0] - 1) / im->vsamp[0];
  const int cb = upsampled(p0 + n0, pw1, dw, dh, hf, vf, x, y) - 128;
  const int cr = upsampled(p0 + n0 + n1, pw1, dw, dh, hf, vf, x, y) - 128;
  // jdcolor.c build_ycc_rgb_table: SCALEBITS 16, ONE_HALF 32768, FIX(v) = (int)(v * 65536 + 0.5)
  const int r = Y + ((91881 * cr + 32768) >> 16);
  const int gch = Y + ((-22554 * cb + 32768 + (-46802 * cr)) >> 16);
  const int bch = Y + ((116130 * cb + 32768) >> 16);
  o[0] = clamp255(r); o[1] = clamp255(gch); o[2] = clamp255(bch);
}

// ---- progressive entropy decode (jdphuff.c) -----------------------------------------------------------------------------
// One lane walks one chain: its scans in file order, each with the sequential BitReader above.  Chains write disjoint
// coefficients (the packer's partition), so the lanes need no synchronisation; the coefficient buffer is zeroed first
// because the scans accumulate into it.
__device__ __forceinline__ uint32_t get_bits(BitReader& br, int n) {          // n raw bits, 0 <= n <= 16
  ensure32(br);
  const uint32_t v = n ? (uint32_t)(br.acc >> (64 - n)) : 0u;
  br.acc <<= n;
  br.n -= n;
  return v;
}
// one Huffman symbol, no value bits (the refinement scans read their own)
__device__ __forceinline__ int decode_symbol(BitReader& br, const gnc_jpeg_huff_t* t) {
  ensure32(br);
  const uint32_t w = (uint32_t)(br.acc >> 32);
  const uint32_t look = t->look[w >> (32 - kLook)];
  int len, sym;
  if (look) {
    len = (int)(look >> 8); sym = (int)(look & 0xff);
  } else {
    len = kLook + 1;
    int32_t code = (int32_t)(w >> (32 - len));
    while (len <= 16 && code > t->maxcode[len]) { ++len; code = (int32_t)(w >> (32 - len)); }
    if (len > 16) { len = 16; sym = 0; }
    else sym = t->vals[(code + t->valoff[len]) & 0xff];
  }
  br.acc <<= len;
  br.n -= len;
  return sym;
}
// zigzag index -> natural position, with libjpeg's clamp (jpeg_natural_order's 16 extra entries are all 63): a corrupt
// run cannot leave the block
__device__ __forceinline__ int natural(int k) { return c_natural[k < 63 ? k : 63]; }

// decode_mcu_AC_refine's correction bit for a nonzero coefficient
__device__ __forceinline__ void refine_coef(BitReader& br, int16_t* c, int p1) {
  const int v = *c;
  if (get_bits(br, 1) && (v & p1) == 0) *c = (int16_t)(v >= 0 ? v + p1 : v - p1);
}

// start of component c's plane in the image's coefficients (the planes are MCU-padded and follow each other)
__device__ __forceinline__ int64_t comp_base(const gnc_jpeg_image_t* im, int c) {
  int64_t b = 0;
  for (int cc = 0; cc < c; ++cc) b += (int64_t)im->mcu_x * im->hsamp[cc] * im->mcu_y * im->vsamp[cc] * 64;
  return b;
}

__device__ __forceinline__ void decode_progressive_scan(const uint8_t* __restrict__ stream, const gnc_jpeg_image_t* im,
                                                        const gnc_jpeg_scan_t* __restrict__ sc,
                                                        const gnc_jpeg_huff_t* __restrict__ tables, int16_t* __restrict__ coef) {
  BitReader br;
  br.p = stream + sc->offset;
  br.end = br.p + sc->bytes;
  br.acc = 0; br.n = 0; br.marker = false;
  int16_t* cimg = coef + im->coef_offset;
  const int Ss = sc->Ss, Se = sc->Se, Ah = sc->Ah, Al = sc->Al, ns = sc->ncomp;
  const int p1 = 1 << Al;
  const bool interleaved = ns > 1;
  // a single-component scan covers the component's own ceil(W h / 8 hmax) x ceil(H v / 8 vmax) blocks, raster order
  const int c0 = sc->comp[0];
  const int nx = interleaved ? im->mcu_x : (im->width * im->hsamp[c0] + 8 * im->hsamp[0] - 1) / (8 * im->hsamp[0]);
  const int ny = interleaved ? im->mcu_y : (im->height * im->vsamp[c0] + 8 * im->vsamp[0] - 1) / (8 * im->vsamp[0]);
  int16_t* const plane0 = cimg + comp_base(im, c0);
  const int bw0 = im->mcu_x * im->hsamp[c0];
  const gnc_jpeg_huff_t* act = tables + sc->ac_tab;
  int pred0 = 0, pred1 = 0, pred2 = 0;
  int eobrun = 0;
  const int restart = sc->restart_interval;
  int to_restart = restart;
  auto block = [&](int16_t* blk, int j, int& pred) {
    if (Ss == 0) {
      if (Ah == 0) {                                   // DC first: prediction, << Al
        int v;
        decode_pair<true>(br, tables + sc->dc_tab[j], v);
        pred += v;
        blk[0] = (int16_t)((unsigned)pred << Al);
      } else if (get_bits(br, 1)) {                    // DC refine: one raw bit
        blk[0] = (int16_t)(blk[0] | p1);
      }
      return;
    }
    if (Ah == 0) {                                     // AC first: EOBRUN, run / size symbols, << Al
      if (eobrun) { --eobrun; return; }
      for (int k = Ss; k <= Se; ++k) {
        int v;
        const int sym = decode_pair<false>(br, act, v);
        const int r = sym >> 4;
        if (sym & 15) {
          k += r;
          blk[natural(k)] = (int16_t)((unsigned)v << Al);
        } else if (r == 15) {
          k += 15;
        } else {
          eobrun = (1 << r) - 1 + (int)get_bits(br, r);
          break;
        }
      }
      return;
    }
    int k = Ss;                                        // AC refine
    if (eobrun == 0) {
      for (; k <= Se; ++k) {
        const int sym = decode_symbol(br, act);
        int r = sym >> 4, s = 0;
        if (sym & 15) {
          s = get_bits(br, 1) ? p1 : -p1;              // a new coefficient: +-(1 << Al)
        } else if (r != 15) {
          eobrun = (1 << r) + (int)get_bits(br, r);
          break;
        }
        do {                                           // the run passes over nonzero coefficients: correction bits
          int16_t* c = blk + natural(k);
          if (*c != 0) refine_coef(br, c, p1);
          else if (--r < 0) break;
          ++k;
        } while (k <= Se);
        if (s) blk[natural(k)] = (int16_t)s;
      }
    }
    if (eobrun > 0) {                                  // inside an end-of-band run: correction bits only
      for (; k <= Se; ++k) {
        int16_t* c = blk + natural(k);
        if (*c != 0) refine_coef(br, c, p1);
      }
      --eobrun;
    }
  };
  for (int y = 0; y < ny; ++y) {
    for (int x = 0; x < nx; ++x) {
      if (restart && to_restart == 0) {
        // byte-align, step over the RSTn marker, reset the predictions and the end-of-band run (jdphuff.c process_restart)
        br.acc = 0; br.n = 0;
        if (br.marker) { br.p += 2; br.marker = false; }
        else {
          while (br.p + 1 < br.end && !(br.p[0] == 0xFF && br.p[1] >= 0xD0 && br.p[1] <= 0xD7)) ++br.p;
          br.p += 2;
        }
        pred0 = pred1 = pred2 = 0;
        eobrun = 0;
        to_restart = restart;
      }
      if (interleaved) {                               // DC scans only: the frame's MCUs, as decode_sequential walks them
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          if (j >= ns) break;
          const int c = sc->comp[j], h = im->hsamp[c], v = im->vsamp[c];
          int16_t* plane = cimg + comp_base(im, c);
          const int bw = im->mcu_x * h;
          for (int by = 0; by < v; ++by)
            for (int bx = 0; bx < h; ++bx)
              block(plane + ((int64_t)(y * v + by) * bw + (x * h + bx)) * 64, j, j == 0 ? pred0 : (j == 1 ? pred1 : pred2));
        }
      } else {
        block(plane0 + ((int64_t)y * bw0 + x) * 64, 0, pred0);
      }
      if (restart) --to_restart;
    }
  }
}

// chains longest first: warp w takes chains [w * per_warp, (w + 1) * per_warp), one per lane.  (128, 1): without the
// minimum ptxas held the kernel to 64 registers and spilled
__global__ void __launch_bounds__(128, 1) jpeg_progressive_kernel(const uint8_t* __restrict__ stream,
                                                               const gnc_jpeg_image_t* __restrict__ frames,
                                                               const gnc_jpeg_scan_t* __restrict__ scans,
                                                               const gnc_jpeg_chain_t* __restrict__ chains, int n_chains,
                                                               const gnc_jpeg_huff_t* __restrict__ tables,
                                                               int16_t* __restrict__ coef, int per_warp) {
  const int lane = threadIdx.x & 31;
  if (lane >= per_warp) return;
  const int64_t ch = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * per_warp + lane;
  if (ch >= n_chains) return;
  const int first = chains[ch].first_scan, last = first + chains[ch].n_scans;
  for (int s = first; s < last; ++s) decode_progressive_scan(stream, frames + scans[s].image, scans + s, tables, coef);
}

// ---- host: marker parser ----------------------------------------------------------------------------------------------
static int build_huff(const uint8_t* bits /*[17], bits[0] unused*/, const uint8_t* vals, int nvals, gnc_jpeg_huff_t* t) {
  memset(t, 0, sizeof(*t));
  int huffsize[257];
  int p = 0;
  for (int l = 1; l <= 16; ++l) {
    const int n = bits[l];
    if (p + n > 256) return 1;
    for (int i = 0; i < n; ++i) huffsize[p++] = l;
  }
  if (p != nvals) return 1;
  huffsize[p] = 0;
  int huffcode[257];
  int code = 0, si = huffsize[0];
  for (int i = 0; i < p;) {
    while (i < p && huffsize[i] == si) huffcode[i++] = code++;
    if (code > (1 << si)) return 1;
    code <<= 1;
    ++si;
  }
  int q = 0;
  for (int l = 1; l <= 16; ++l) {
    if (bits[l]) {
      t->valoff[l] = q - huffcode[q];
      q += bits[l];
      t->maxcode[l] = huffcode[q - 1];
    } else {
      t->maxcode[l] = -1;
      t->valoff[l] = 0;
    }
  }
  t->maxcode[17] = 0x7fffffff;
  for (int i = 0; i < p; ++i) t->vals[i] = vals[i];
  q = 0;
  for (int l = 1; l <= kLook; ++l) {
    for (int i = 0; i < bits[l]; ++i, ++q) {
      const int first = huffcode[q] << (kLook - l);
      for (int k = 0; k < (1 << (kLook - l)); ++k) t->look[first + k] = (uint16_t)((l << 8) | vals[q]);
    }
  }
  return 0;
}

// ---- host: progressive marker parser ----------------------------------------------------------------------------------
// oracle/jpeg_progressive.py parse_progressive restates these rules; tests/test_jpeg_progressive.py holds the two to the same files.
struct ProgFile {
  std::vector<gnc_jpeg_scan_t> scans;    // file order; offsets relative to the file, tables indices into `tables`
  std::vector<int> chain;                // chain of each scan, numbered by first scan
  std::vector<gnc_jpeg_huff_t> tables;
  int n_chains = 0;
};

// libjpeg (jdhuff.c jpeg_make_d_derived_tbl) rejects tables that overflow a code length or use an all-ones code
static bool huff_codes_ok(const uint8_t* bits /*[17]*/) {
  int code = 0;
  for (int l = 1; l <= 16; ++l) {
    code += bits[l];
    if (code >= (1 << l)) return false;
    code <<= 1;
  }
  return true;
}

static int parse_progressive(const uint8_t* data, int64_t size, gnc_jpeg_image_t* out, ProgFile& pf) {
  constexpr int UNSUP = GNC_JPEG_UNSUPPORTED;
  memset(out, 0, sizeof(*out));
  pf.scans.clear(); pf.chain.clear(); pf.tables.clear(); pf.n_chains = 0;
  if (!data || size < 4 || data[0] != 0xFF || data[1] != 0xD8) return UNSUP;
  uint8_t dht_bits[8][17];
  uint8_t dht_vals[8][256];
  int dht_n[8];
  int dht_emitted[8];                                   // index in pf.tables of the slot's current definition, -1: none yet
  bool dht_set[8] = {false, false, false, false, false, false, false, false};
  uint16_t qcur[4][64];
  bool q_set[4] = {false, false, false, false};
  bool latched[3] = {false, false, false};
  int comp_id[3] = {0, 0, 0};
  int coef_bits[3][64];                                 // jdinput.c coef_bits: -1 never coded, else the current Al
  bool have_sof = false;
  int adobe_transform = -1, dri = 0;
  int64_t pos = 2;
  for (;;) {
    if (pos + 2 > size || data[pos] != 0xFF) return UNSUP;
    const int m = data[pos + 1];
    if (m == 0xFF) { ++pos; continue; }                 // fill byte
    pos += 2;
    if (m == 0xD9) break;                               // EOI
    if (m == 0xD8 || (m >= 0xD0 && m <= 0xD7) || m == 0x01) continue;
    if (pos + 2 > size) return UNSUP;
    const int64_t len = ((int64_t)data[pos] << 8) | data[pos + 1];
    if (len < 2 || pos + len > size) return UNSUP;
    const uint8_t* seg = data + pos + 2;
    const int64_t n = len - 2;
    if (m == 0xC2) {                                    // progressive, Huffman
      if (have_sof || n < 6 || seg[0] != 8) return UNSUP;
      out->height = (seg[1] << 8) | seg[2];
      out->width = (seg[3] << 8) | seg[4];
      out->ncomp = seg[5];
      if ((out->ncomp != 1 && out->ncomp != 3) || out->width <= 0 || out->height <= 0 || n < 6 + 3 * out->ncomp) return UNSUP;
      for (int c = 0; c < out->ncomp; ++c) {
        comp_id[c] = seg[6 + 3 * c];
        out->hsamp[c] = seg[7 + 3 * c] >> 4;
        out->vsamp[c] = seg[7 + 3 * c] & 15;
        out->qtab[c] = seg[8 + 3 * c];
        if (out->qtab[c] > 3 || out->hsamp[c] < 1 || out->hsamp[c] > 4 || out->vsamp[c] < 1 || out->vsamp[c] > 4) return UNSUP;
        for (int d = 0; d < c; ++d)
          if (comp_id[d] == comp_id[c]) return UNSUP;
        for (int k = 0; k < 64; ++k) coef_bits[c][k] = -1;
      }
      have_sof = true;
    } else if (m >= 0xC0 && m <= 0xCF && m != 0xC4 && m != 0xC8) {
      return UNSUP;                                     // sequential, lossless, arithmetic, hierarchical
    } else if (m == 0xDC) {
      return UNSUP;                                     // DNL
    } else if (m == 0xC4) {                             // DHT: a new definition of the slot
      int64_t i = 0;
      while (i < n) {
        if (i + 17 > n) return UNSUP;
        const int tc = seg[i] >> 4, th = seg[i] & 15;
        if (tc > 1 || th > 3) return UNSUP;
        const int slot = tc * 4 + th;
        int cnt = 0;
        dht_bits[slot][0] = 0;
        for (int l = 1; l <= 16; ++l) { dht_bits[slot][l] = seg[i + l]; cnt += seg[i + l]; }
        if (cnt > 256 || i + 17 + cnt > n || !huff_codes_ok(dht_bits[slot])) return UNSUP;
        memcpy(dht_vals[slot], seg + i + 17, (size_t)cnt);
        if (tc == 0)
          for (int k = 0; k < cnt; ++k)
            if (dht_vals[slot][k] > 15) return UNSUP;
        dht_n[slot] = cnt;
        dht_set[slot] = true;
        dht_emitted[slot] = -1;
        i += 17 + cnt;
      }
    } else if (m == 0xDB) {                             // DQT
      int64_t i = 0;
      while (i < n) {
        const int pq = seg[i] >> 4, tq = seg[i] & 15;
        if (tq > 3 || pq > 1 || i + 1 + 64 * (pq + 1) > n) return UNSUP;
        for (int k = 0; k < 64; ++k) {
          const int v = pq ? ((seg[i + 1 + 2 * k] << 8) | seg[i + 2 + 2 * k]) : seg[i + 1 + k];
          qcur[tq][h_natural[k]] = (uint16_t)v;
        }
        q_set[tq] = true;
        i += 1 + 64 * (pq + 1);
      }
    } else if (m == 0xDD) {                             // DRI: in force for the scans that follow
      if (n < 2) return UNSUP;
      dri = (seg[0] << 8) | seg[1];
    } else if (m == 0xEE) {
      if (n >= 12 && memcmp(seg, "Adobe", 5) == 0) adobe_transform = seg[11];
    } else if (m == 0xDA) {                             // SOS
      if (!have_sof) return UNSUP;
      const int nc = out->ncomp;
      if (nc == 3) {                                    // the baseline parser's colour space and layout rules
        if (adobe_transform == 0) return UNSUP;
        if (adobe_transform < 0 && comp_id[0] == 'R' && comp_id[1] == 'G' && comp_id[2] == 'B') return UNSUP;
        if (out->hsamp[1] != 1 || out->vsamp[1] != 1 || out->hsamp[2] != 1 || out->vsamp[2] != 1) return UNSUP;
        const int h = out->hsamp[0], v = out->vsamp[0];
        if (!((h == 1 && v == 1) || (h == 2 && v == 1) || (h == 2 && v == 2))) return UNSUP;
      }
      const int ns = n >= 1 ? seg[0] : 0;
      if (ns < 1 || ns > nc || n < 1 + 2 * ns + 3) return UNSUP;
      gnc_jpeg_scan_t sc;
      memset(&sc, 0, sizeof(sc));
      sc.ncomp = ns;
      int td[3] = {0, 0, 0}, ta = 0;
      for (int j = 0; j < ns; ++j) {
        int c = 0;
        while (c < nc && comp_id[c] != seg[1 + 2 * j]) ++c;
        if (c == nc || (j > 0 && c <= sc.comp[j - 1])) return UNSUP;       // known components, in frame order
        sc.comp[j] = c;
        td[j] = seg[2 + 2 * j] >> 4;
        ta = seg[2 + 2 * j] & 15;
      }
      sc.Ss = seg[1 + 2 * ns]; sc.Se = seg[2 + 2 * ns]; sc.Ah = seg[3 + 2 * ns] >> 4; sc.Al = seg[3 + 2 * ns] & 15;
      // jdphuff.c start_pass_phuff_decoder: what it rejects, and what it only warns about
      if (sc.Ss == 0) {
        if (sc.Se != 0) return UNSUP;
      } else if (sc.Ss > sc.Se || sc.Se > 63 || ns != 1) {
        return UNSUP;
      }
      if ((sc.Ah != 0 && sc.Al != sc.Ah - 1) || sc.Al > 13) return UNSUP;
      for (int j = 0; j < ns; ++j) {
        int* cb = coef_bits[sc.comp[j]];
        if (sc.Ss != 0 && cb[0] < 0) return UNSUP;    // AC before the component's first DC scan
        for (int k = sc.Ss; k <= sc.Se; ++k) {
          if (sc.Ah == 0 ? cb[k] != -1 : cb[k] != sc.Ah) return UNSUP;
          cb[k] = sc.Al;
        }
      }
      // Huffman tables as they stand now (a DHT before almost every scan is the rule)
      auto emit = [&](int slot) -> int {
        if (!dht_set[slot]) return -1;
        if (dht_emitted[slot] < 0) {
          if ((int)pf.tables.size() >= GNC_JPEG_MAX_TABLES) return -1;
          pf.tables.emplace_back();
          if (build_huff(dht_bits[slot], dht_vals[slot], dht_n[slot], &pf.tables.back())) return -1;
          dht_emitted[slot] = (int)pf.tables.size() - 1;
        }
        return dht_emitted[slot];
      };
      if (sc.Ss == 0 && sc.Ah == 0) {
        for (int j = 0; j < ns; ++j)
          if (td[j] > 3 || (sc.dc_tab[j] = emit(td[j])) < 0) return UNSUP;
      }
      if (sc.Ss != 0 && (ta > 3 || (sc.ac_tab = emit(4 + ta)) < 0)) return UNSUP;
      // quantisation tables are latched at a component's first scan (jdinput.c latch_quant_tables)
      for (int j = 0; j < ns; ++j) {
        const int c = sc.comp[j];
        if (latched[c]) continue;
        if (!q_set[out->qtab[c]]) return UNSUP;
        memcpy(out->quant[c], qcur[out->qtab[c]], sizeof(out->quant[c]));
        latched[c] = true;
      }
      sc.restart_interval = dri;
      sc.offset = pos + len;
      // the entropy-coded segment runs to the next marker that is not RSTn / stuffing / fill; it must exist
      int64_t e = sc.offset;
      while (e + 1 < size) {
        if (data[e] == 0xFF && data[e + 1] != 0 && !(data[e + 1] >= 0xD0 && data[e + 1] <= 0xD7) && data[e + 1] != 0xFF) break;
        ++e;
      }
      if (e + 1 >= size) return UNSUP;
      sc.bytes = e - sc.offset;
      if ((int)pf.scans.size() >= GNC_JPEG_MAX_SCANS) return UNSUP;
      pf.scans.push_back(sc);
      pos = e;
      continue;
    }
    pos += len;
  }
  if (pf.scans.empty()) return UNSUP;
  // jdcoefct.c smoothing_ok (libjpeg-turbo >= 2.1, SAVED_COEFS = 10): a DC never coded, or an AC coefficient 1..9 of
  // some component not fully refined, and libjpeg smooths across blocks - out of scope
  for (int c = 0; c < out->ncomp; ++c) {
    if (coef_bits[c][0] < 0) return UNSUP;
    for (int k = 1; k < 10; ++k)
      if (coef_bits[c][k] != 0) return UNSUP;
  }
  if (out->ncomp == 1) out->hsamp[0] = out->vsamp[0] = 1;          // a single component is never interleaved
  for (int c = 0; c < out->ncomp; ++c) out->qtab[c] = c;           // quant[c] = component c's latched table
  out->mcu_x = (out->width + 8 * out->hsamp[0] - 1) / (8 * out->hsamp[0]);
  out->mcu_y = (out->height + 8 * out->vsamp[0] - 1) / (8 * out->vsamp[0]);
  int64_t blocks = 0;
  for (int c = 0; c < out->ncomp; ++c) blocks += (int64_t)out->mcu_x * out->hsamp[c] * out->mcu_y * out->vsamp[c];
  out->n_blocks = blocks;
  out->plane_bytes = blocks * 64;
  // chains: union of scans that write a common (component, coefficient); numbered by first scan
  const int S = (int)pf.scans.size();
  std::vector<int> parent((size_t)S);
  for (int s = 0; s < S; ++s) parent[s] = s;
  auto root = [&](int s) { while (parent[s] != s) s = parent[s] = parent[parent[s]]; return s; };
  int last[3][64];
  for (int c = 0; c < 3; ++c)
    for (int k = 0; k < 64; ++k) last[c][k] = -1;
  for (int s = 0; s < S; ++s) {
    const gnc_jpeg_scan_t& sc = pf.scans[s];
    for (int j = 0; j < sc.ncomp; ++j)
      for (int k = sc.Ss; k <= sc.Se; ++k) {
        int& l = last[sc.comp[j]][k];
        if (l >= 0) parent[root(l)] = root(s);
        l = s;
      }
  }
  pf.chain.assign((size_t)S, -1);
  std::vector<int> id_of_root((size_t)S, -1);
  for (int s = 0; s < S; ++s) {
    int& id = id_of_root[root(s)];
    if (id < 0) id = pf.n_chains++;
    pf.chain[s] = id;
  }
  return GNC_OK;
}

}  // namespace jpeg
}  // namespace gnc

using namespace gnc;

extern "C" {

int gnc_jpeg_parse(const uint8_t* data, int64_t size, gnc_jpeg_image_t* out) {
  if (!data || !out || size < 4) return GNC_JPEG_UNSUPPORTED;
  memset(out, 0, sizeof(*out));
  if (data[0] != 0xFF || data[1] != 0xD8) return GNC_JPEG_UNSUPPORTED;
  uint8_t dht_bits[8][17];
  uint8_t dht_vals[8][256];
  int dht_n[8];
  bool dht_set[8] = {false, false, false, false, false, false, false, false};
  bool q_set[4] = {false, false, false, false};
  int comp_id[3] = {0, 0, 0};
  bool have_sof = false;
  int adobe_transform = -1;
  int64_t pos = 2;
  while (pos + 4 <= size) {
    if (data[pos] != 0xFF) return GNC_JPEG_UNSUPPORTED;
    int m = data[pos + 1];
    if (m == 0xFF) { ++pos; continue; }                   // fill byte
    pos += 2;
    if (m == 0xD8 || (m >= 0xD0 && m <= 0xD7) || m == 0x01) continue;
    if (m == 0xD9) return GNC_JPEG_UNSUPPORTED;           // EOI before a scan
    const int64_t len = ((int64_t)data[pos] << 8) | data[pos + 1];
    if (len < 2 || pos + len > size) return GNC_JPEG_UNSUPPORTED;
    const uint8_t* seg = data + pos + 2;
    const int64_t n = len - 2;
    if (m == 0xC0 || m == 0xC1) {                         // baseline / extended sequential, Huffman
      if (n < 6 || seg[0] != 8) return GNC_JPEG_UNSUPPORTED;
      out->height = (seg[1] << 8) | seg[2];
      out->width = (seg[3] << 8) | seg[4];
      out->ncomp = seg[5];
      if ((out->ncomp != 1 && out->ncomp != 3) || out->width <= 0 || out->height <= 0 || n < 6 + 3 * out->ncomp) return GNC_JPEG_UNSUPPORTED;
      for (int c = 0; c < out->ncomp; ++c) {
        comp_id[c] = seg[6 + 3 * c];
        out->hsamp[c] = seg[7 + 3 * c] >> 4;
        out->vsamp[c] = seg[7 + 3 * c] & 15;
        out->qtab[c] = seg[8 + 3 * c];
        if (out->qtab[c] > 3) return GNC_JPEG_UNSUPPORTED;
      }
      have_sof = true;
    } else if (m >= 0xC2 && m <= 0xCF && m != 0xC4 && m != 0xC8 && m != 0xCC) {
      return GNC_JPEG_UNSUPPORTED;                        // progressive, lossless, arithmetic, hierarchical
    } else if (m == 0xCC) {
      return GNC_JPEG_UNSUPPORTED;
    } else if (m == 0xC4) {                               // DHT
      int64_t i = 0;
      while (i + 17 <= n) {
        const int tc = seg[i] >> 4, th = seg[i] & 15;
        if (tc > 1 || th > 3) return GNC_JPEG_UNSUPPORTED;
        const int slot = tc * 4 + th;
        int cnt = 0;
        dht_bits[slot][0] = 0;
        for (int l = 1; l <= 16; ++l) { dht_bits[slot][l] = seg[i + l]; cnt += seg[i + l]; }
        if (cnt > 256 || i + 17 + cnt > n) return GNC_JPEG_UNSUPPORTED;
        memcpy(dht_vals[slot], seg + i + 17, (size_t)cnt);
        dht_n[slot] = cnt;
        dht_set[slot] = true;
        i += 17 + cnt;
      }
    } else if (m == 0xDB) {                               // DQT
      int64_t i = 0;
      while (i < n) {
        const int pq = seg[i] >> 4, tq = seg[i] & 15;
        if (tq > 3 || pq > 1 || i + 1 + 64 * (pq + 1) > n) return GNC_JPEG_UNSUPPORTED;
        for (int k = 0; k < 64; ++k) {
          const int v = pq ? ((seg[i + 1 + 2 * k] << 8) | seg[i + 2 + 2 * k]) : seg[i + 1 + k];
          out->quant[tq][jpeg::h_natural[k]] = (uint16_t)v;
        }
        q_set[tq] = true;
        i += 1 + 64 * (pq + 1);
      }
    } else if (m == 0xDD) {                               // DRI
      if (n < 2) return GNC_JPEG_UNSUPPORTED;
      out->restart_interval = (seg[0] << 8) | seg[1];
    } else if (m == 0xEE) {                               // Adobe: the colour transform flag
      if (n >= 12 && memcmp(seg, "Adobe", 5) == 0) adobe_transform = seg[11];
    } else if (m == 0xDA) {                               // SOS
      if (!have_sof || n < 1 || seg[0] != out->ncomp || n < 1 + 2 * out->ncomp + 3) return GNC_JPEG_UNSUPPORTED;
      for (int c = 0; c < out->ncomp; ++c) {
        if (seg[1 + 2 * c] != comp_id[c]) return GNC_JPEG_UNSUPPORTED;      // one interleaved scan in frame order
        out->dc_tab[c] = seg[2 + 2 * c] >> 4;
        out->ac_tab[c] = seg[2 + 2 * c] & 15;
        if (out->dc_tab[c] > 3 || out->ac_tab[c] > 3) return GNC_JPEG_UNSUPPORTED;
        if (!dht_set[out->dc_tab[c]] || !dht_set[4 + out->ac_tab[c]] || !q_set[out->qtab[c]]) return GNC_JPEG_UNSUPPORTED;
      }
      // colour space as libjpeg guesses it: 3 components are YCbCr unless an Adobe marker says RGB (transform 0) or
      // the component ids spell R, G, B
      if (out->ncomp == 3) {
        if (adobe_transform == 0) return GNC_JPEG_UNSUPPORTED;
        if (adobe_transform < 0 && comp_id[0] == 'R' && comp_id[1] == 'G' && comp_id[2] == 'B') return GNC_JPEG_UNSUPPORTED;
        // chroma: both at 1 x 1, luma 1 x 1, 2 x 1 or 2 x 2 (4:4:4, 4:2:2, 4:2:0)
        if (out->hsamp[1] != 1 || out->vsamp[1] != 1 || out->hsamp[2] != 1 || out->vsamp[2] != 1) return GNC_JPEG_UNSUPPORTED;
        const int h = out->hsamp[0], v = out->vsamp[0];
        if (!((h == 1 && v == 1) || (h == 2 && v == 1) || (h == 2 && v == 2))) return GNC_JPEG_UNSUPPORTED;
      } else {
        out->hsamp[0] = out->vsamp[0] = 1;                // a single component is never interleaved: 1 x 1 blocks
      }
      for (int s = 0; s < 8; ++s)
        if (dht_set[s] && jpeg::build_huff(dht_bits[s], dht_vals[s], dht_n[s], &out->huff[s])) return GNC_JPEG_UNSUPPORTED;
      out->mcu_x = (out->width + 8 * out->hsamp[0] - 1) / (8 * out->hsamp[0]);
      out->mcu_y = (out->height + 8 * out->vsamp[0] - 1) / (8 * out->vsamp[0]);
      out->scan_offset = pos + len;
      // the entropy-coded segment runs to the next marker that is not RSTn / stuffing; a second scan is not supported
      int64_t e = out->scan_offset;
      while (e + 1 < size) {
        if (data[e] == 0xFF && data[e + 1] != 0 && !(data[e + 1] >= 0xD0 && data[e + 1] <= 0xD7) && data[e + 1] != 0xFF) break;
        ++e;
      }
      if (e + 1 >= size) e = size;
      else if (data[e + 1] != 0xD9) return GNC_JPEG_UNSUPPORTED;            // something other than EOI follows the scan
      out->scan_bytes = e - out->scan_offset;
      int64_t blocks = 0, plane = 0;
      for (int c = 0; c < out->ncomp; ++c) {
        const int64_t nb = (int64_t)out->mcu_x * out->hsamp[c] * out->mcu_y * out->vsamp[c];
        blocks += nb;
        plane += nb * 64;
      }
      out->n_blocks = blocks;
      out->plane_bytes = plane;
      return GNC_OK;
    }
    pos += len;
  }
  return GNC_JPEG_UNSUPPORTED;
}

// HOST: descriptors + byte stream of a whole batch in one call (parse and copies spread over `threads` host threads).
// Files the device decoder does not cover are left out; index_out lists the files that are in, in order.
int gnc_jpeg_pack(const uint8_t* const* datas, const int64_t* sizes, int n, int threads, uint8_t* stream_out,
                  int64_t stream_capacity, gnc_jpeg_image_t* infos_out, int32_t* index_out, int64_t* totals) {
  GNC_REQUIRE(n >= 0 && (n == 0 || (datas && sizes && stream_out && infos_out && index_out)) && totals, "jpeg_pack: bad arguments");
  std::vector<int> ok((size_t)n, 0);
  const int nt = threads < 1 ? 1 : (threads > 32 ? 32 : threads);
  auto parallel = [&](auto&& fn) {
    if (nt == 1 || n < 8) { for (int i = 0; i < n; ++i) fn(i); return; }
    std::vector<std::thread> pool;
    for (int t = 0; t < nt; ++t) pool.emplace_back([&, t]() { for (int i = t; i < n; i += nt) fn(i); });
    for (auto& th : pool) th.join();
  };
  parallel([&](int i) { ok[i] = gnc_jpeg_parse(datas[i], sizes[i], infos_out + i) == GNC_OK; });
  int m = 0;
  int64_t off = 0, blocks = 0, plane = 0, pixels = 0;
  std::vector<int64_t> dst((size_t)n, 0);
  for (int i = 0; i < n; ++i) {
    if (!ok[i]) continue;
    if (m != i) memcpy(infos_out + m, infos_out + i, sizeof(gnc_jpeg_image_t));
    gnc_jpeg_image_t& d = infos_out[m];
    dst[m] = off;
    d.scan_offset += off;
    d.block_offset = blocks; d.coef_offset = 64 * blocks; d.plane_offset = plane; d.pixel_offset = pixels;
    index_out[m] = i;
    off += sizes[i]; blocks += d.n_blocks; plane += d.plane_bytes; pixels += (int64_t)d.width * d.height;
    ++m;
  }
  GNC_REQUIRE(off <= stream_capacity, "jpeg_pack: stream buffer too small");
  const int mm = m;
  {
    const int n_keep = mm;
    auto copy = [&](int j) { memcpy(stream_out + dst[j], datas[index_out[j]], (size_t)sizes[index_out[j]]); };
    if (nt == 1 || n_keep < 8) { for (int j = 0; j < n_keep; ++j) copy(j); }
    else {
      std::vector<std::thread> pool;
      for (int t = 0; t < nt; ++t) pool.emplace_back([&, t]() { for (int j = t; j < n_keep; j += nt) copy(j); });
      for (auto& th : pool) th.join();
    }
  }
  totals[0] = mm; totals[1] = off; totals[2] = blocks; totals[3] = plane; totals[4] = pixels;
  return GNC_OK;
}

static int g_jpeg_sequential = 0;

// Debug: 1 = the entropy stage always runs its sequential form (one thread per image).  Same coefficients.
int gnc_debug_jpeg_sequential(int on) {
  g_jpeg_sequential = on;                         // bit 0: sequential form; bit 1: print the synchronisation rounds of images 0-2
  return GNC_OK;
}

int64_t gnc_jpeg_scratch_bytes(int64_t stream_bytes, int B) { return stream_bytes + 16 * (int64_t)(B > 0 ? B : 0) + 64; }

int gnc_jpeg_decode_rgb_u8(const uint8_t* stream, const gnc_jpeg_image_t* infos, int B, int64_t total_blocks,
                           int64_t total_pixels, int16_t* coef, uint8_t* planes, uint8_t* out, uint8_t* scratch,
                           gnc_stream_t stream_) {
  GNC_REQUIRE(B >= 0 && total_blocks >= 0 && total_pixels >= 0, "jpeg_decode: bad sizes");
  if (B == 0) return GNC_OK;
  GNC_REQUIRE(stream && infos && coef && planes && out, "jpeg_decode: null pointer");
  cudaStream_t st = (cudaStream_t)stream_;
  cudaError_t e = cudaMemsetAsync(coef, 0, (size_t)total_blocks * 64 * sizeof(int16_t), st);
  if (e != cudaSuccess) return fail(GNC_ECUDA, "jpeg memset: %s", cudaGetErrorString(e));
  jpeg::jpeg_huffman_kernel<<<(unsigned)ceil_div<int>(B, jpeg::kHuffWarps), 32 * jpeg::kHuffWarps,
                              jpeg::kHuffWarps * 8 * sizeof(gnc_jpeg_huff_t), st>>>(stream, infos, B, coef, scratch,
                                                                                    g_jpeg_sequential);
  if (int rc = check_launch("jpeg_huffman_kernel")) return rc;
  jpeg::jpeg_idct_kernel<<<(unsigned)ceil_div<int64_t>(total_blocks, 128), 128, 0, st>>>(infos, B, coef, planes, total_blocks);
  if (int rc = check_launch("jpeg_idct_kernel")) return rc;
  jpeg::jpeg_color_kernel<<<(unsigned)ceil_div<int64_t>(total_pixels, 256), 256, 0, st>>>(infos, B, planes, out, total_pixels);
  return check_launch("jpeg_color_kernel");
}

int gnc_jpeg_pack_progressive(const uint8_t* const* datas, const int64_t* sizes, int n, int threads, uint8_t* stream_out,
                              int64_t stream_capacity, gnc_jpeg_image_t* frames_out, int32_t* index_out,
                              gnc_jpeg_scan_t* scans_out, int64_t scan_capacity, gnc_jpeg_chain_t* chains_out,
                              int64_t chain_capacity, gnc_jpeg_huff_t* tables_out, int64_t table_capacity, int64_t* totals) {
  GNC_REQUIRE(n >= 0 && (n == 0 || (datas && sizes && stream_out && frames_out && index_out && scans_out && chains_out && tables_out)) &&
                  totals, "jpeg_pack_progressive: bad arguments");
  std::vector<jpeg::ProgFile> files((size_t)n);
  std::vector<int> ok((size_t)n, 0);
  const int nt = threads < 1 ? 1 : (threads > 32 ? 32 : threads);
  auto parallel = [&](int count, auto&& fn) {
    if (nt == 1 || count < 8) { for (int i = 0; i < count; ++i) fn(i); return; }
    std::vector<std::thread> pool;
    for (int t = 0; t < nt; ++t) pool.emplace_back([&, t]() { for (int i = t; i < count; i += nt) fn(i); });
    for (auto& th : pool) th.join();
  };
  parallel(n, [&](int i) { ok[i] = jpeg::parse_progressive(datas[i], sizes[i], frames_out + i, files[i]) == GNC_OK; });
  // offsets of the files that are in
  struct ChainRef { int64_t bytes; int file, chain; };
  std::vector<ChainRef> refs;
  std::vector<int64_t> dst, table_base;
  int m = 0;
  int64_t off = 0, blocks = 0, plane = 0, pixels = 0, n_scans = 0, n_tables = 0;
  for (int i = 0; i < n; ++i) {
    if (!ok[i]) continue;
    if (m != i) memcpy(frames_out + m, frames_out + i, sizeof(gnc_jpeg_image_t));
    gnc_jpeg_image_t& d = frames_out[m];
    d.block_offset = blocks; d.coef_offset = 64 * blocks; d.plane_offset = plane; d.pixel_offset = pixels;
    index_out[m] = i;
    dst.push_back(off);
    table_base.push_back(n_tables);
    const jpeg::ProgFile& pf = files[i];
    std::vector<int64_t> chain_bytes((size_t)pf.n_chains, 0);
    for (size_t s = 0; s < pf.scans.size(); ++s) chain_bytes[pf.chain[s]] += pf.scans[s].bytes;
    for (int c = 0; c < pf.n_chains; ++c) refs.push_back({chain_bytes[c], m, c});
    off += sizes[i]; blocks += d.n_blocks; plane += d.plane_bytes; pixels += (int64_t)d.width * d.height;
    n_scans += (int64_t)pf.scans.size(); n_tables += (int64_t)pf.tables.size();
    ++m;
  }
  GNC_REQUIRE(off <= stream_capacity, "jpeg_pack_progressive: stream buffer too small");
  GNC_REQUIRE(n_scans <= scan_capacity && (int64_t)refs.size() <= chain_capacity && n_tables <= table_capacity,
              "jpeg_pack_progressive: scan / chain / table buffer too small");
  // chains longest first across the batch, each chain's scans together in file order
  std::stable_sort(refs.begin(), refs.end(), [](const ChainRef& a, const ChainRef& b) { return a.bytes > b.bytes; });
  int64_t s_out = 0;
  for (size_t r = 0; r < refs.size(); ++r) {
    const jpeg::ProgFile& pf = files[index_out[refs[r].file]];
    chains_out[r].first_scan = (int32_t)s_out;
    chains_out[r].bytes = refs[r].bytes;
    for (size_t s = 0; s < pf.scans.size(); ++s) {
      if (pf.chain[s] != refs[r].chain) continue;
      gnc_jpeg_scan_t sc = pf.scans[s];
      sc.image = refs[r].file;
      sc.offset += dst[refs[r].file];
      for (int j = 0; j < 3; ++j) sc.dc_tab[j] += (int32_t)table_base[refs[r].file];
      sc.ac_tab += (int32_t)table_base[refs[r].file];
      scans_out[s_out++] = sc;
    }
    chains_out[r].n_scans = (int32_t)(s_out - chains_out[r].first_scan);
  }
  parallel(m, [&](int j) {
    const jpeg::ProgFile& pf = files[index_out[j]];
    memcpy(stream_out + dst[j], datas[index_out[j]], (size_t)sizes[index_out[j]]);
    if (!pf.tables.empty()) memcpy(tables_out + table_base[j], pf.tables.data(), pf.tables.size() * sizeof(gnc_jpeg_huff_t));
  });
  totals[0] = m; totals[1] = off; totals[2] = blocks; totals[3] = plane; totals[4] = pixels;
  totals[5] = n_scans; totals[6] = (int64_t)refs.size(); totals[7] = n_tables;
  return GNC_OK;
}

// One chain per warp by default: the lanes of a warp sit in different scans and procedures, so a warp's lanes take turns;
// 512 files of 375 x 500 (2 048 chains) decode 6.5 x faster with one chain per warp than with 32
// (profiles/r06_jpeg_progressive_bench.txt).
static int g_jpeg_chains_per_warp = 1;

int gnc_debug_jpeg_chains_per_warp(int n) {
  g_jpeg_chains_per_warp = (n >= 1 && n <= 32) ? n : 1;
  return GNC_OK;
}

int gnc_jpeg_decode_progressive_rgb_u8(const uint8_t* stream, const gnc_jpeg_image_t* frames, int B,
                                       const gnc_jpeg_scan_t* scans, const gnc_jpeg_chain_t* chains, int n_chains,
                                       const gnc_jpeg_huff_t* tables, int64_t total_blocks, int64_t total_pixels,
                                       int16_t* coef, uint8_t* planes, uint8_t* out, gnc_stream_t stream_) {
  GNC_REQUIRE(B >= 0 && n_chains >= 0 && total_blocks >= 0 && total_pixels >= 0, "jpeg_decode_progressive: bad sizes");
  if (B == 0) return GNC_OK;
  GNC_REQUIRE(stream && frames && scans && chains && tables && coef && planes && out, "jpeg_decode_progressive: null pointer");
  cudaStream_t st = (cudaStream_t)stream_;
  cudaError_t e = cudaMemsetAsync(coef, 0, (size_t)total_blocks * 64 * sizeof(int16_t), st);
  if (e != cudaSuccess) return fail(GNC_ECUDA, "jpeg memset: %s", cudaGetErrorString(e));
  if (n_chains > 0) {
    const int per_warp = g_jpeg_chains_per_warp;
    const int64_t warps = ceil_div<int64_t>(n_chains, per_warp);
    jpeg::jpeg_progressive_kernel<<<(unsigned)ceil_div<int64_t>(warps, 4), 128, 0, st>>>(stream, frames, scans, chains, n_chains,
                                                                                      tables, coef, per_warp);
    if (int rc = check_launch("jpeg_progressive_kernel")) return rc;
  }
  jpeg::jpeg_idct_kernel<<<(unsigned)ceil_div<int64_t>(total_blocks, 128), 128, 0, st>>>(frames, B, coef, planes, total_blocks);
  if (int rc = check_launch("jpeg_idct_kernel")) return rc;
  jpeg::jpeg_color_kernel<<<(unsigned)ceil_div<int64_t>(total_pixels, 256), 256, 0, st>>>(frames, B, planes, out, total_pixels);
  return check_launch("jpeg_color_kernel");
}

}  // extern "C"
