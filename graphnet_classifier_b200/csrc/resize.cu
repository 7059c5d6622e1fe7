// Pillow-exact bicubic resize of RGB uint8 images on the device (input staging of the graph builders).
//
// The reference turns every image into its working resolution with PIL:
//   Image.open(path).convert('RGB').resize((r, r))         utils/image_to_graph/image_to_graph_optimized.py:65-70
// i.e. Pillow's ImagingResample with the BICUBIC filter: a separable two-pass convolution (horizontal first),
// an 8-bit intermediate image, per-output-pixel coefficient windows computed in double precision and
// quantised to 22-bit fixed point, int32 accumulation from the rounding constant 1 << 21, arithmetic shift,
// clamp to a byte.  Everything after the coefficient tables is integer arithmetic, so the device result is
// bit-identical to Pillow's; the tables themselves are computed on the host with the same double-precision
// expressions (gnc_resize_bicubic_coeffs).
//
// HBM-bound byte work: per image 3*H*W bytes in, 3*OH*OW bytes out; the intermediate [H, OW, 3] image is
// written and re-read once (it stays in L2 for typical photo sizes).
//   horizontal pass: one CTA per source row - the row is staged in shared memory with 16-byte loads, every
//                    thread produces 4 consecutive output bytes (one 32-bit store);
//   vertical pass:   one thread per 4 consecutive bytes of an output row, taps read as 32-bit words
//                    (adjacent threads -> adjacent words), weights are warp-uniform.
#include "common.cuh"

namespace gnc {
namespace rsz {

constexpr int kPrecisionBits = 32 - 8 - 2;
constexpr int kThreads = 128;

__device__ __forceinline__ uint32_t clip8(int v) {
  v >>= kPrecisionBits;
  return (uint32_t)min(max(v, 0), 255);
}

// src rows: [rows] x row_bytes = 3 * W, row r of image b at src + b * image_stride + y * pitch
__global__ void __launch_bounds__(kThreads) resize_h_kernel(const uint8_t* __restrict__ src, int H, int W, long long pitch,
                                                             long long image_stride, int OW, const int32_t* __restrict__ bounds,
                                                             const int32_t* __restrict__ kk, int ksize, uint8_t* __restrict__ dst) {
  extern __shared__ __align__(16) uint8_t s_row[];
  const long long row = blockIdx.x;
  const long long b = row / H;
  const int y = (int)(row - b * H);
  const uint8_t* g = src + b * image_stride + (long long)y * pitch;
  const int nbytes = 3 * W;
  // stage the row: shared offset keeps the global address's 16-byte phase, so that the aligned middle part
  // moves as 128-bit words
  const int phase = (int)(reinterpret_cast<uintptr_t>(g) & 15u);
  uint8_t* s = s_row + phase;
  const int head = min(nbytes, (16 - phase) & 15);
  const int nvec = (nbytes - head) >> 4;
  for (int i = threadIdx.x; i < head; i += kThreads) s[i] = g[i];
  const uint4* gv = reinterpret_cast<const uint4*>(g + head);
  uint4* sv = reinterpret_cast<uint4*>(s + head);
  for (int i = threadIdx.x; i < nvec; i += kThreads) sv[i] = __ldg(gv + i);
  for (int i = head + (nvec << 4) + threadIdx.x; i < nbytes; i += kThreads) s[i] = g[i];
  __syncthreads();

  const int obytes = 3 * OW;
  uint8_t* out = dst + row * (long long)obytes;
  const bool word_ok = (reinterpret_cast<uintptr_t>(out) & 3u) == 0;
  for (int o4 = threadIdx.x * 4; o4 < obytes; o4 += kThreads * 4) {
    uint32_t packed = 0;
    const int n_out = min(4, obytes - o4);
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      if (t < n_out) {
        const int o = o4 + t;
        const int xx = o / 3, c = o - 3 * xx;
        const int xmin = __ldg(bounds + 2 * xx), n = __ldg(bounds + 2 * xx + 1);
        const int32_t* k = kk + (long long)xx * ksize;
        const uint8_t* p = s + 3 * xmin + c;
        int acc = 1 << (kPrecisionBits - 1);
        for (int x = 0; x < n; ++x) acc += (int)p[3 * x] * __ldg(k + x);
        packed |= clip8(acc) << (8 * t);
      }
    }
    if (n_out == 4 && word_ok) {
      *reinterpret_cast<uint32_t*>(out + o4) = packed;
    } else {
      for (int t = 0; t < n_out; ++t) out[o4 + t] = (uint8_t)(packed >> (8 * t));
    }
  }
}

// Stages `nrows` consecutive source rows (flattened over images) in shared memory, one warp per row (rows warp,
// warp + 4, ...), so the per-row address set-up is paid by 32 lanes only.  Each row keeps the 16-byte phase of its
// global address (s_phase[r]), so that its aligned middle part moves as 128-bit words.
__device__ __forceinline__ void stage_rows(const uint8_t* __restrict__ src, int H, long long pitch, long long image_stride,
                                           long long row0, int nrows, int nbytes, int row_stride, int* s_phase, uint8_t* s_rows) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long img0 = row0 / H;                        // one division per thread, then carried
  const int y0 = (int)(row0 - img0 * H);
  for (int r = warp; r < nrows; r += kThreads / 32) {
    long long img = img0;
    int y = y0 + r;
    while (y >= H) { y -= H; ++img; }
    const uint8_t* g = src + img * image_stride + (long long)y * pitch;
    const int phase = (int)(reinterpret_cast<uintptr_t>(g) & 15u);
    if (lane == 0) s_phase[r] = phase;
    uint8_t* s = s_rows + (long long)r * row_stride + phase;
    const int head = min(nbytes, (16 - phase) & 15);
    const int nvec = (nbytes - head) >> 4;
    if (lane < head) s[lane] = g[lane];
    const uint4* gv = reinterpret_cast<const uint4*>(g + head);
    uint4* sv = reinterpret_cast<uint4*>(s + head);
    for (int i = lane; i < nvec; i += 32) sv[i] = __ldg(gv + i);
    const int tail0 = head + (nvec << 4);
    if (tail0 + lane < nbytes) s[tail0 + lane] = g[tail0 + lane];
  }
}

// Register-resident form of the horizontal pass (windows of at most KMAX taps): a CTA stages R source rows, thread
// xx keeps its KMAX weights in registers and walks its byte window of every staged row as 32-bit shared-memory
// words (funnel-shifted to the window's byte phase) - one LDS per 4 multiply-adds instead of one per multiply-add,
// and the weight table is read once per R rows instead of once per row.
template <int KMAX>
__global__ void __launch_bounds__(kThreads) resize_h_reg_kernel(const uint8_t* __restrict__ src, int H, int W, long long pitch,
                                                                 long long image_stride, int OW, const int32_t* __restrict__ bounds,
                                                                 const int32_t* __restrict__ kk, int ksize, uint8_t* __restrict__ dst,
                                                                 long long total_rows, int R, int row_stride) {
  extern __shared__ __align__(16) uint8_t s_all[];
  int* s_phase = reinterpret_cast<int*>(s_all);          // [16]: 16-byte phase of each staged row's global address
  uint8_t* s_rows = s_all + 64;
  const long long row0 = (long long)blockIdx.x * R;
  const int nrows = (int)min((long long)R, total_rows - row0);
  const int nbytes = 3 * W;
  stage_rows(src, H, pitch, image_stride, row0, nrows, nbytes, row_stride, s_phase, s_rows);
  __syncthreads();
  const int xx = blockIdx.y * kThreads + threadIdx.x;
  if (xx >= OW) return;
  const int xmin = __ldg(bounds + 2 * xx), n = __ldg(bounds + 2 * xx + 1);
  int kreg[KMAX];
#pragma unroll
  for (int x = 0; x < KMAX; ++x) kreg[x] = x < n ? __ldg(kk + (long long)xx * ksize + x) : 0;
  constexpr int kWinBytes = 3 * KMAX;
  constexpr int kWords = (kWinBytes + 3) / 4;
  for (int r = 0; r < nrows; ++r) {
    const long long row = row0 + r;
    const int a = s_phase[r] + 3 * xmin;                  // first byte of the window inside the staged row
    const uint32_t* wp = reinterpret_cast<const uint32_t*>(s_rows + (long long)r * row_stride) + (a >> 2);
    const int sh = (a & 3) * 8;
    uint32_t wd[kWords + 1];
#pragma unroll
    for (int j = 0; j <= kWords; ++j) wd[j] = wp[j];      // bytes past the window meet zero weights
    int acc[3] = {1 << (kPrecisionBits - 1), 1 << (kPrecisionBits - 1), 1 << (kPrecisionBits - 1)};
#pragma unroll
    for (int j = 0; j < kWords; ++j) {
      const uint32_t w = __funnelshift_r(wd[j], wd[j + 1], sh);
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int i = 4 * j + t;
        if (i < kWinBytes) acc[i % 3] += (int)__byte_perm(w, 0u, 0x4440u + t) * kreg[i / 3];
      }
    }
    uint8_t* out = dst + row * (3LL * OW) + 3 * xx;
    out[0] = (uint8_t)clip8(acc[0]);
    out[1] = (uint8_t)clip8(acc[1]);
    out[2] = (uint8_t)clip8(acc[2]);
  }
}

template <int KMAX>
static int launch_h_reg(const uint8_t* src, int64_t B, int H, int W, int64_t pitch, int64_t istride, int OW, const int32_t* bounds,
                        const int32_t* kk, int ksize, uint8_t* dst, cudaStream_t st) {
  constexpr int kSmemCap = 64 * 1024;
  const int slack = 3 * KMAX + 16 + 64;
  const int row_stride = (3 * W + 16 + 15) & ~15;
  int R = (kSmemCap - slack) / row_stride;
  if (R < 1) return -1;                                   // row too wide for this form: the caller falls back
  if (R > 16) R = 16;
  const size_t smem = (size_t)R * row_stride + slack;
  static SmemAttrOnce smem_attr;
  if (int rc_attr = smem_attr.ensure(resize_h_reg_kernel<KMAX>, kSmemCap, "resize_bicubic")) return rc_attr;
  const long long rows = B * (long long)H;
  dim3 grid((unsigned)ceil_div(rows, (long long)R), (unsigned)ceil_div(OW, kThreads));
  resize_h_reg_kernel<KMAX><<<grid, kThreads, smem, st>>>(src, H, W, pitch, istride, OW, bounds, kk, ksize, dst, rows, R, row_stride);
  return check_launch("resize_h_reg_kernel");
}

// Long windows (down-scaling by more than 8: more than 33 taps): the window is walked in chunks of KCH taps; a chunk's
// weights are loaded once and applied to all RMAX staged rows, whose accumulators stay in registers across chunks.
template <int KCH, int RMAX>
__global__ void __launch_bounds__(kThreads) resize_h_long_kernel(const uint8_t* __restrict__ src, int H, int W, long long pitch,
                                                                  long long image_stride, int OW, const int32_t* __restrict__ bounds,
                                                                  const int32_t* __restrict__ kk, int ksize, uint8_t* __restrict__ dst,
                                                                  long long total_rows, int R, int row_stride) {
  extern __shared__ __align__(16) uint8_t s_all[];
  int* s_phase = reinterpret_cast<int*>(s_all);
  uint8_t* s_rows = s_all + 64;
  const long long row0 = (long long)blockIdx.x * R;
  const int nrows = (int)min((long long)R, total_rows - row0);
  stage_rows(src, H, pitch, image_stride, row0, nrows, 3 * W, row_stride, s_phase, s_rows);
  __syncthreads();
  const int xx = blockIdx.y * kThreads + threadIdx.x;
  if (xx >= OW) return;
  const int xmin = __ldg(bounds + 2 * xx), n = __ldg(bounds + 2 * xx + 1);
  const int32_t* k = kk + (long long)xx * ksize;
  constexpr int kWinBytes = 3 * KCH;
  constexpr int kWords = (kWinBytes + 3) / 4;
  int acc[RMAX][3];
#pragma unroll
  for (int r = 0; r < RMAX; ++r) acc[r][0] = acc[r][1] = acc[r][2] = 1 << (kPrecisionBits - 1);
  for (int c0 = 0; c0 < n; c0 += KCH) {
    int kreg[KCH];
#pragma unroll
    for (int x = 0; x < KCH; ++x) kreg[x] = c0 + x < n ? __ldg(k + c0 + x) : 0;
#pragma unroll
    for (int r = 0; r < RMAX; ++r) {
      if (r < nrows) {
        const int a = s_phase[r] + 3 * (xmin + c0);
        const uint32_t* wp = reinterpret_cast<const uint32_t*>(s_rows + (long long)r * row_stride) + (a >> 2);
        const int sh = (a & 3) * 8;
        uint32_t wd[kWords + 1];
#pragma unroll
        for (int j = 0; j <= kWords; ++j) wd[j] = wp[j];
#pragma unroll
        for (int j = 0; j < kWords; ++j) {
          const uint32_t w = __funnelshift_r(wd[j], wd[j + 1], sh);
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const int i = 4 * j + t;
            if (i < kWinBytes) acc[r][i % 3] += (int)__byte_perm(w, 0u, 0x4440u + t) * kreg[i / 3];
          }
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < RMAX; ++r) {
    if (r < nrows) {
      uint8_t* out = dst + (row0 + r) * (3LL * OW) + 3 * xx;
      out[0] = (uint8_t)clip8(acc[r][0]);
      out[1] = (uint8_t)clip8(acc[r][1]);
      out[2] = (uint8_t)clip8(acc[r][2]);
    }
  }
}

static int launch_h_long(const uint8_t* src, int64_t B, int H, int W, int64_t pitch, int64_t istride, int OW, const int32_t* bounds,
                         const int32_t* kk, int ksize, uint8_t* dst, cudaStream_t st) {
  constexpr int KCH = 32, RMAX = 4, kSmemCap = 96 * 1024;
  const int slack = 3 * KCH + 16 + 64;
  const int row_stride = (3 * W + 16 + 15) & ~15;
  int R = (kSmemCap - slack) / row_stride;
  if (R < 1) return -1;                                   // wider than ~32 000 pixels: the generic kernel
  if (R > RMAX) R = RMAX;
  const size_t smem = (size_t)R * row_stride + slack;
  static SmemAttrOnce smem_attr;
  if (int rc_attr = smem_attr.ensure(resize_h_long_kernel<KCH, RMAX>, kSmemCap, "resize_bicubic")) return rc_attr;
  const long long rows = B * (long long)H;
  dim3 grid((unsigned)ceil_div(rows, (long long)R), (unsigned)ceil_div(OW, kThreads));
  resize_h_long_kernel<KCH, RMAX><<<grid, kThreads, smem, st>>>(src, H, W, pitch, istride, OW, bounds, kk, ksize, dst, rows, R, row_stride);
  return check_launch("resize_h_long_kernel");
}

// One output word of the vertical pass: n_out (1..4) bytes at `out` from the n taps p, p + pitch, ... weighted by k.
__device__ __forceinline__ void v_taps(const uint8_t* p, long long pitch, const int32_t* k, int n, int n_out, uint8_t* out) {
  int a0, a1, a2, a3;
  a0 = a1 = a2 = a3 = 1 << (kPrecisionBits - 1);
  const bool word_in = n_out == 4 && ((reinterpret_cast<uintptr_t>(p) | (uintptr_t)pitch) & 3u) == 0;
  if (word_in) {
    for (int y = 0; y < n; ++y) {
      const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(p + (long long)y * pitch));
      const int c = __ldg(k + y);
      a0 += (int)(w & 255u) * c;
      a1 += (int)((w >> 8) & 255u) * c;
      a2 += (int)((w >> 16) & 255u) * c;
      a3 += (int)(w >> 24) * c;
    }
  } else {
    for (int y = 0; y < n; ++y) {
      const uint8_t* q = p + (long long)y * pitch;
      const int c = __ldg(k + y);
      a0 += (int)q[0] * c;
      if (n_out > 1) a1 += (int)q[1] * c;
      if (n_out > 2) a2 += (int)q[2] * c;
      if (n_out > 3) a3 += (int)q[3] * c;
    }
  }
  const uint32_t packed = clip8(a0) | (clip8(a1) << 8) | (clip8(a2) << 16) | (clip8(a3) << 24);
  if (n_out == 4 && (reinterpret_cast<uintptr_t>(out) & 3u) == 0) {
    *reinterpret_cast<uint32_t*>(out) = packed;
  } else {
    for (int t = 0; t < n_out; ++t) out[t] = (uint8_t)(packed >> (8 * t));
  }
}

// src: [B] images of H rows x row_bytes (pitch / image_stride in bytes); dst: [B, OH, row_bytes] contiguous.
// One thread per 32-bit word of the output (flattened over rows, so narrow rows still fill the CTAs).
__global__ void __launch_bounds__(kThreads) resize_v_kernel(const uint8_t* __restrict__ src, int row_bytes, long long pitch,
                                                             long long image_stride, int OH, long long n_rows,
                                                             const int32_t* __restrict__ bounds, const int32_t* __restrict__ kk,
                                                             int ksize, uint8_t* __restrict__ dst) {
  const int wpr = (row_bytes + 3) >> 2;              // words per output row
  const long long idx = (long long)blockIdx.x * kThreads + threadIdx.x;
  const long long orow = idx / wpr;                  // b * OH + yy
  if (orow >= n_rows) return;
  const int o4 = (int)(idx - orow * wpr) * 4;
  const long long b = orow / OH;
  const int yy = (int)(orow - b * OH);
  const int ymin = __ldg(bounds + 2 * yy), n = __ldg(bounds + 2 * yy + 1);
  const int32_t* k = kk + (long long)yy * ksize;
  const uint8_t* p = src + b * image_stride + (long long)ymin * pitch + o4;
  uint8_t* out = dst + orow * (long long)row_bytes + o4;
  const int n_out = min(4, row_bytes - o4);
  v_taps(p, pitch, k, n, n_out, out);
}

// Vertical pass, 16 output bytes per thread (rows and pitches that are multiples of 16 bytes: any OW % 16 == 0):
// one 128-bit load and one weight per tap feed 16 multiply-adds.
__global__ void __launch_bounds__(kThreads) resize_v16_kernel(const uint8_t* __restrict__ src, int row_bytes, long long pitch,
                                                               long long image_stride, int OH, long long n_rows,
                                                               const int32_t* __restrict__ bounds, const int32_t* __restrict__ kk,
                                                               int ksize, uint8_t* __restrict__ dst) {
  const int vpr = row_bytes >> 4;                    // 16-byte vectors per output row
  const long long idx = (long long)blockIdx.x * kThreads + threadIdx.x;
  const long long orow = idx / vpr;
  if (orow >= n_rows) return;
  const int o16 = (int)(idx - orow * vpr) * 16;
  const long long b = orow / OH;
  const int yy = (int)(orow - b * OH);
  const int ymin = __ldg(bounds + 2 * yy), n = __ldg(bounds + 2 * yy + 1);
  const int32_t* k = kk + (long long)yy * ksize;
  const uint8_t* p = src + b * image_stride + (long long)ymin * pitch + o16;
  int acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 1 << (kPrecisionBits - 1);
#pragma unroll 2
  for (int y = 0; y < n; ++y, p += pitch) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
    const int c = __ldg(k + y);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] += (int)__byte_perm(w[i >> 2], 0u, 0x4440u + (i & 3)) * c;
  }
  uint32_t o[4];
#pragma unroll
  for (int j = 0; j < 4; ++j)
    o[j] = clip8(acc[4 * j]) | (clip8(acc[4 * j + 1]) << 8) | (clip8(acc[4 * j + 2]) << 16) | (clip8(acc[4 * j + 3]) << 24);
  *reinterpret_cast<uint4*>(dst + orow * (long long)row_bytes + o16) = make_uint4(o[0], o[1], o[2], o[3]);
}

// ---- ragged batches: every image has its own H x W, all go to OH x OW ---------------------------------------------
// Three launches whatever the number of shapes: the coefficient tables of every image, the horizontal pass over the
// rows of the images whose width changes, the vertical pass over all n * OH output rows.

// Pillow's bicubic kernel (a = -0.5) in double precision, each operation rounded on its own as the host code's
// (built with -ffp-contract=off): nvcc would otherwise fuse the multiply-adds and the tables would differ.
__device__ __forceinline__ double bicubic_filter_dev(double x) {
  if (x < 0.0) x = -x;
  if (x < 1.0) return __dadd_rn(__dmul_rn(__dmul_rn(__dsub_rn(__dmul_rn(1.5, x), 2.5), x), x), 1.0);
  if (x < 2.0) return __dmul_rn(__dsub_rn(__dmul_rn(__dadd_rn(__dmul_rn(__dsub_rn(x, 5.0), x), 8.0), x), 4.0), -0.5);
  return 0.0;
}

// One thread per output position of either axis of every image (n x (OW + OH) threads): the bounds and kk rows of
// gnc_resize_bicubic_coeffs, at the image's workspace offsets.  Axes that keep their size (ksize 0) have no table.
__global__ void __launch_bounds__(kThreads) resize_ragged_tables_kernel(const gnc_resize_image_t* __restrict__ images,
                                                                         long long n, int OH, int OW, int32_t* __restrict__ tables) {
  const long long idx = (long long)blockIdx.x * kThreads + threadIdx.x;
  const long long i = idx / (OW + OH);
  if (i >= n) return;
  int xx = (int)(idx - i * (OW + OH));
  const gnc_resize_image_t* im = images + i;
  int in_size, out_size, ksize;
  long long tab;
  if (xx < OW) {
    in_size = im->width, out_size = OW, ksize = im->ksize_x, tab = im->tab_x;
  } else {
    xx -= OW;
    in_size = im->height, out_size = OH, ksize = im->ksize_y, tab = im->tab_y;
  }
  if (ksize == 0) return;
  const double scale = __ddiv_rn((double)in_size, (double)out_size);
  const double filterscale = scale < 1.0 ? 1.0 : scale;
  const double support = __dmul_rn(2.0, filterscale);
  const double ss = __ddiv_rn(1.0, filterscale);
  const double center = __dadd_rn(0.0, __dmul_rn(__dadd_rn((double)xx, 0.5), scale));
  int xmin = (int)__dadd_rn(__dsub_rn(center, support), 0.5);
  if (xmin < 0) xmin = 0;
  int xmax = (int)__dadd_rn(__dadd_rn(center, support), 0.5);
  if (xmax > in_size) xmax = in_size;
  xmax -= xmin;
  int32_t* bounds = tables + tab;
  int32_t* k = bounds + 2 * out_size + (long long)xx * ksize;
  double ww = 0.0;
  for (int x = 0; x < xmax; ++x)
    ww = __dadd_rn(ww, bicubic_filter_dev(__dmul_rn(__dadd_rn(__dsub_rn((double)(x + xmin), center), 0.5), ss)));
  for (int x = 0; x < xmax; ++x) {
    double v = bicubic_filter_dev(__dmul_rn(__dadd_rn(__dsub_rn((double)(x + xmin), center), 0.5), ss));
    if (ww != 0.0) v = __ddiv_rn(v, ww);
    v = __dmul_rn(v, (double)(1 << kPrecisionBits));
    k[x] = v < 0 ? (int)__dadd_rn(-0.5, v) : (int)__dadd_rn(0.5, v);
  }
  for (int x = xmax; x < ksize; ++x) k[x] = 0;
  bounds[2 * xx] = xmin;
  bounds[2 * xx + 1] = xmax;
}

// Horizontal pass, one CTA per row of tmp [h_rows, OW, 3]: the rows of the images whose width changes, image after
// image (tmp_row = running row count).  The row's image is the last one whose tmp_row is <= the row: images that
// contribute no rows share their tmp_row with the next image, which the search then prefers.
__global__ void __launch_bounds__(kThreads) resize_ragged_h_kernel(const gnc_resize_image_t* __restrict__ images, int n, int OW,
                                                                    const int32_t* __restrict__ tables, uint8_t* __restrict__ tmp) {
  extern __shared__ __align__(16) uint8_t s_row[];
  __shared__ int s_image;
  const long long row = blockIdx.x;
  if (threadIdx.x == 0) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (images[mid].tmp_row <= row) lo = mid;
      else hi = mid - 1;
    }
    s_image = lo;
  }
  __syncthreads();
  const gnc_resize_image_t* im = images + s_image;
  const uint8_t* g = im->src + (row - im->tmp_row) * im->pitch;
  const int nbytes = 3 * im->width;
  // the shared copy keeps the row's 16-byte phase, so that its aligned middle part moves as 128-bit words
  const int phase = (int)(reinterpret_cast<uintptr_t>(g) & 15u);
  uint8_t* s = s_row + phase;
  const int head = min(nbytes, (16 - phase) & 15);
  const int nvec = (nbytes - head) >> 4;
  for (int i = threadIdx.x; i < head; i += kThreads) s[i] = g[i];
  const uint4* gv = reinterpret_cast<const uint4*>(g + head);
  uint4* sv = reinterpret_cast<uint4*>(s + head);
  for (int i = threadIdx.x; i < nvec; i += kThreads) sv[i] = __ldg(gv + i);
  for (int i = head + (nvec << 4) + threadIdx.x; i < nbytes; i += kThreads) s[i] = g[i];
  __syncthreads();

  const int ksize = im->ksize_x;
  const int32_t* bounds = tables + im->tab_x;
  const int32_t* kk = bounds + 2 * OW;
  uint8_t* out = tmp + row * (3LL * OW);
  for (int xx = threadIdx.x; xx < OW; xx += kThreads) {
    const int xmin = __ldg(bounds + 2 * xx), nt = __ldg(bounds + 2 * xx + 1);
    const int32_t* k = kk + (long long)xx * ksize;
    const uint8_t* p = s + 3 * xmin;
    int a0, a1, a2;
    a0 = a1 = a2 = 1 << (kPrecisionBits - 1);
    for (int x = 0; x < nt; ++x) {
      const int c = __ldg(k + x);
      a0 += (int)p[3 * x] * c;
      a1 += (int)p[3 * x + 1] * c;
      a2 += (int)p[3 * x + 2] * c;
    }
    out[3 * xx] = (uint8_t)clip8(a0);
    out[3 * xx + 1] = (uint8_t)clip8(a1);
    out[3 * xx + 2] = (uint8_t)clip8(a2);
  }
}

// Vertical pass, one thread per 32-bit word of dst [n, OH, OW, 3].  An image reads its rows from tmp when its width
// changed, else from its source; an image whose height is already OH copies row yy.
__global__ void __launch_bounds__(kThreads) resize_ragged_v_kernel(const gnc_resize_image_t* __restrict__ images, long long n_rows,
                                                                    int OH, int OW, const int32_t* __restrict__ tables,
                                                                    const uint8_t* __restrict__ tmp, uint8_t* __restrict__ dst) {
  const int row_bytes = 3 * OW;
  const int wpr = (row_bytes + 3) >> 2;
  const long long idx = (long long)blockIdx.x * kThreads + threadIdx.x;
  const long long orow = idx / wpr;                  // i * OH + yy
  if (orow >= n_rows) return;
  const int o4 = (int)(idx - orow * wpr) * 4;
  const long long i = orow / OH;
  const int yy = (int)(orow - i * OH);
  const gnc_resize_image_t* im = images + i;
  const bool from_tmp = im->ksize_x != 0;
  const uint8_t* src = from_tmp ? tmp + im->tmp_row * (long long)row_bytes : im->src;
  const long long pitch = from_tmp ? (long long)row_bytes : im->pitch;
  const int ksize = im->ksize_y;
  uint8_t* out = dst + orow * (long long)row_bytes + o4;
  const int n_out = min(4, row_bytes - o4);
  if (ksize == 0) {
    const uint8_t* p = src + (long long)yy * pitch + o4;
    for (int t = 0; t < n_out; ++t) out[t] = p[t];
    return;
  }
  const int32_t* bounds = tables + im->tab_y;
  const int ymin = __ldg(bounds + 2 * yy), n = __ldg(bounds + 2 * yy + 1);
  v_taps(src + (long long)ymin * pitch + o4, pitch, bounds + 2 * OH + (long long)yy * ksize, n, n_out, out);
}

// ---- coefficient tables (host; Pillow's precompute_coeffs + normalize_coeffs_8bpc, full box) --------------------
static inline double bicubic_filter(double x) {
  const double a = -0.5;
  if (x < 0.0) x = -x;
  if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
  if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
  return 0.0;
}

static int ksize_of(int in_size, int out_size) {
  double filterscale = (double)in_size / out_size;
  if (filterscale < 1.0) filterscale = 1.0;
  const double support = 2.0 * filterscale;
  return (int)ceil(support) * 2 + 1;
}

}  // namespace rsz
}  // namespace gnc

using namespace gnc;

extern "C" int gnc_resize_bicubic_ksize(int in_size, int out_size) {
  if (in_size <= 0 || out_size <= 0) return 0;
  return rsz::ksize_of(in_size, out_size);
}

extern "C" int gnc_resize_bicubic_coeffs(int in_size, int out_size, int32_t* bounds, int32_t* kk) {
  GNC_REQUIRE(in_size > 0 && out_size > 0 && bounds && kk, "resize_bicubic_coeffs: bad arguments");
  const double scale = (double)in_size / out_size;
  double filterscale = scale;
  if (filterscale < 1.0) filterscale = 1.0;
  const double support = 2.0 * filterscale;
  const int ksize = (int)ceil(support) * 2 + 1;
  const double ss = 1.0 / filterscale;
  for (int xx = 0; xx < out_size; ++xx) {
    const double center = 0.0 + (xx + 0.5) * scale;
    int xmin = (int)(center - support + 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = (int)(center + support + 0.5);
    if (xmax > in_size) xmax = in_size;
    xmax -= xmin;
    int32_t* k = kk + (long long)xx * ksize;
    double ww = 0.0;
    // two passes over the window: Pillow stores the raw weights, sums them, then normalises
    for (int x = 0; x < xmax; ++x) ww += rsz::bicubic_filter((x + xmin - center + 0.5) * ss);
    for (int x = 0; x < xmax; ++x) {
      double v = rsz::bicubic_filter((x + xmin - center + 0.5) * ss);
      if (ww != 0.0) v /= ww;
      v *= (double)(1 << rsz::kPrecisionBits);
      k[x] = v < 0 ? (int)(-0.5 + v) : (int)(0.5 + v);
    }
    for (int x = xmax; x < ksize; ++x) k[x] = 0;
    bounds[2 * xx] = xmin;
    bounds[2 * xx + 1] = xmax;
  }
  return GNC_OK;
}

extern "C" int gnc_resize_bicubic_u8(const uint8_t* src, int64_t B, int H, int W, int64_t src_pitch, int64_t src_image_stride,
                                     int OH, int OW, const int32_t* bounds_x, const int32_t* kk_x, int ksize_x,
                                     const int32_t* bounds_y, const int32_t* kk_y, int ksize_y, uint8_t* tmp, uint8_t* dst,
                                     gnc_stream_t stream) {
  GNC_REQUIRE(src && dst && B >= 0 && H > 0 && W > 0 && OH > 0 && OW > 0, "resize_bicubic: bad arguments");
  GNC_REQUIRE(src_pitch >= 3LL * W && src_image_stride >= (int64_t)H * src_pitch, "resize_bicubic: pitch / image stride too small");
  GNC_REQUIRE((W == OW) == (bounds_x == nullptr) && (W == OW || (kk_x && ksize_x > 0)), "resize_bicubic: horizontal tables must be given exactly when the width changes");
  GNC_REQUIRE((H == OH) == (bounds_y == nullptr) && (H == OH || (kk_y && ksize_y > 0)), "resize_bicubic: vertical tables must be given exactly when the height changes");
  GNC_REQUIRE(B * (int64_t)(H > OH ? H : OH) < (1LL << 31), "resize_bicubic: too many rows for one launch");
  if (B == 0) return GNC_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const bool do_h = W != OW, do_v = H != OH;
  if (!do_h && !do_v) {
    cudaError_t e;
    if (src_image_stride == (int64_t)H * src_pitch) {
      e = cudaMemcpy2DAsync(dst, 3LL * W, src, src_pitch, 3LL * W, (size_t)(B * H), cudaMemcpyDeviceToDevice, st);
    } else {
      e = cudaSuccess;
      for (int64_t b = 0; b < B && e == cudaSuccess; ++b)
        e = cudaMemcpy2DAsync(dst + b * 3LL * W * H, 3LL * W, src + b * src_image_stride, src_pitch, 3LL * W, (size_t)H,
                              cudaMemcpyDeviceToDevice, st);
    }
    if (e != cudaSuccess) return fail(GNC_ECUDA, "resize_bicubic: copy: %s", cudaGetErrorString(e));
    return GNC_OK;
  }
  const uint8_t* vsrc = src;
  int64_t vpitch = src_pitch, vstride = src_image_stride;
  if (do_h) {
    GNC_REQUIRE(!do_v || tmp, "resize_bicubic: tmp [B, H, OW, 3] is required when both axes change");
    uint8_t* hdst = do_v ? tmp : dst;
    int rc = -1;                          // -1: the register-resident form does not apply
#define GNC_RSZ_H(K) rsz::launch_h_reg<K>(src, B, H, W, src_pitch, src_image_stride, OW, bounds_x, kk_x, ksize_x, hdst, st)
    if (ksize_x <= 5) rc = GNC_RSZ_H(5);
    else if (ksize_x <= 9) rc = GNC_RSZ_H(9);
    else if (ksize_x <= 13) rc = GNC_RSZ_H(13);
    else if (ksize_x <= 17) rc = GNC_RSZ_H(17);
    else if (ksize_x <= 25) rc = GNC_RSZ_H(25);
    else if (ksize_x <= 33) rc = GNC_RSZ_H(33);
    else rc = rsz::launch_h_long(src, B, H, W, src_pitch, src_image_stride, OW, bounds_x, kk_x, ksize_x, hdst, st);
#undef GNC_RSZ_H
    if (rc < 0) {                         // rows too wide for the staged forms: generic kernel, one row per CTA
      const size_t smem = (size_t)3 * W + 32;
      GNC_REQUIRE(smem <= 200 * 1024, "resize_bicubic: source rows wider than 68 000 pixels are not supported");
      if (smem > 48 * 1024) {             // the attribute is per device: set it on every such launch (cheap, rare path)
        cudaError_t e = cudaFuncSetAttribute(rsz::resize_h_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return fail(GNC_ECUDA, "resize_bicubic: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      }
      rsz::resize_h_kernel<<<(unsigned)(B * H), rsz::kThreads, smem, st>>>(src, H, W, src_pitch, src_image_stride, OW, bounds_x,
                                                                          kk_x, ksize_x, hdst);
      rc = check_launch("resize_h_kernel");
    }
    if (rc != GNC_OK) return rc;
    vsrc = tmp;
    vpitch = 3LL * OW;
    vstride = (int64_t)H * vpitch;
  }
  if (do_v) {
    const int row_bytes = 3 * OW;
    const long long rows = B * (long long)OH;
    const bool vec16 = row_bytes % 16 == 0 && vpitch % 16 == 0 && vstride % 16 == 0 && aligned16(vsrc) && aligned16(dst);
    const long long items = rows * (vec16 ? row_bytes >> 4 : (row_bytes + 3) >> 2);
    const long long blocks = ceil_div(items, (long long)rsz::kThreads);
    GNC_REQUIRE(blocks < (1LL << 31), "resize_bicubic: output too large for one launch");
    if (vec16)
      rsz::resize_v16_kernel<<<(unsigned)blocks, rsz::kThreads, 0, st>>>(vsrc, row_bytes, vpitch, vstride, OH, rows, bounds_y, kk_y,
                                                                        ksize_y, dst);
    else
      rsz::resize_v_kernel<<<(unsigned)blocks, rsz::kThreads, 0, st>>>(vsrc, row_bytes, vpitch, vstride, OH, rows, bounds_y, kk_y,
                                                                      ksize_y, dst);
    int rc = check_launch("resize_v_kernel");
    if (rc != GNC_OK) return rc;
  }
  return GNC_OK;
}

extern "C" int gnc_resize_bicubic_ragged_u8(const gnc_resize_image_t* images, int64_t n, int OH, int OW, int64_t h_rows, int max_w,
                                            int32_t* tables, uint8_t* tmp, uint8_t* dst, gnc_stream_t stream) {
  GNC_REQUIRE(n >= 0 && OH > 0 && OW > 0 && h_rows >= 0 && max_w >= 0, "resize_bicubic_ragged: bad arguments");
  if (n == 0) return GNC_OK;
  GNC_REQUIRE(images && tables && dst, "resize_bicubic_ragged: images, tables and dst are required");
  GNC_REQUIRE(h_rows == 0 || (tmp && max_w > 0), "resize_bicubic_ragged: tmp [h_rows, OW, 3] and max_w are required when a width changes");
  GNC_REQUIRE(n < (1LL << 31) && h_rows < (1LL << 31), "resize_bicubic_ragged: too many images or rows for one launch");
  const size_t smem = (size_t)3 * max_w + 32;
  GNC_REQUIRE(smem <= 200 * 1024, "resize_bicubic_ragged: source rows wider than 68 000 pixels are not supported");
  cudaStream_t st = (cudaStream_t)stream;
  const long long tab_blocks = ceil_div(n * (long long)(OW + OH), (long long)rsz::kThreads);
  const long long v_blocks = ceil_div(n * (long long)OH * ((3LL * OW + 3) >> 2), (long long)rsz::kThreads);
  GNC_REQUIRE(tab_blocks < (1LL << 31) && v_blocks < (1LL << 31), "resize_bicubic_ragged: output too large for one launch");
  rsz::resize_ragged_tables_kernel<<<(unsigned)tab_blocks, rsz::kThreads, 0, st>>>(images, n, OH, OW, tables);
  int rc = check_launch("resize_ragged_tables_kernel");
  if (rc != GNC_OK) return rc;
  if (h_rows > 0) {
    static SmemAttrOnce smem_attr;
    if (smem > 48 * 1024)
      if (int rc_attr = smem_attr.ensure(rsz::resize_ragged_h_kernel, 200 * 1024, "resize_bicubic_ragged")) return rc_attr;
    rsz::resize_ragged_h_kernel<<<(unsigned)h_rows, rsz::kThreads, smem, st>>>(images, (int)n, OW, tables, tmp);
    rc = check_launch("resize_ragged_h_kernel");
    if (rc != GNC_OK) return rc;
  }
  rsz::resize_ragged_v_kernel<<<(unsigned)v_blocks, rsz::kThreads, 0, st>>>(images, n * (long long)OH, OH, OW, tables, tmp, dst);
  return check_launch("resize_ragged_v_kernel");
}
