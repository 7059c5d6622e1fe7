// Dense operators of the GraphNet MLPs (sm_100a, fp32 CUDA-core path).
//
// nn.Linear (+bias, +ReLU) forward, data-gradient and weight-gradient as ONE
// register-tiled 128x128x16 FP32 GEMM template whose operand loaders understand
// "gathered, column-concatenated" matrices (gnc_seg_t), so the reference's
//   cat([x[row], x[col], edge_attr])  (models/GNN.py:58-60 + MetaLayer gathers :146/:215)
//   cat([x, agg])                     (models/GNN.py:100)
// are consumed in place and never materialised.  LayerNorm (+residual) forward /
// backward and the bias / ReLU backward column reductions complete models/MLP.py:24-37.
//
// fp32 FMA keeps the 1e-5 logits/gradients parity bar with two decades of margin
// (SURVEY.md section 0.2: single-pass TF32/BF16 fail it); the tcgen05 3xTF32 path
// replaces this engine tile-for-tile, the layouts here are the ones it consumes.
#include "common.cuh"

namespace gnc {

constexpr int BM = 128;        // output tile rows
constexpr int BN = 128;        // output tile cols
constexpr int BK = 16;         // reduce chunk
constexpr int LDT = BM + 4;    // smem row pitch (floats): 2-way worst-case conflicts on transposing stores
constexpr int kGemmThreads = 256;
constexpr int kMaxSeg = 3;

struct Operand {
  const float* base[kMaxSeg];
  const int32_t* idx[kMaxSeg];
  long long ld[kMaxSeg];
  int start[kMaxSeg + 1];   // prefix sums of widths
  int nseg;
};

struct GemmArgs {
  Operand A, B;
  long long rows;        // output rows   (fwd/dgrad: M;  wgrad: N)
  int cols;              // output cols   (fwd: N; dgrad: K; wgrad: K)
  long long red;         // reduce extent (fwd: K; dgrad: N; wgrad: M)
  long long red_chunk;   // reduce range per blockIdx.z (multiple of BK)
  float* C;
  long long ldc;
  long long c_split_stride;  // wgrad partials: elements between splits
  const float* bias;
  int relu, accumulate, vec_store;
};

// ---- operand loaders ---------------------------------------------------------
// T operand: tile [128 out-rows][BK reduce], source is reduce-contiguous; staged
// transposed into S[k][row].  Row gather (idx) applies to the out-row; segments
// split the reduce dimension.
template <bool FAST>
struct TLoader {
  const Operand& op;
  long long row0, nrows;
  // fast state
  int seg;
  const float* p[2];
  float4 v[2];
  // slow state
  float sv[8];

  __device__ __forceinline__ TLoader(const Operand& o, long long r0, long long nr) : op(o), row0(r0), nrows(nr) {
    seg = -1;
    p[0] = p[1] = nullptr;
  }

  __device__ __forceinline__ void fetch(long long k0, long long red_end) {
    const int t = threadIdx.x;
    if constexpr (FAST) {
      const int rq = t >> 2, kq = t & 3;
      if (seg < 0 || k0 >= op.start[seg + 1]) {
        if (seg < 0) seg = 0;
        while (k0 >= op.start[seg + 1]) ++seg;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const long long r = row0 + rq + 64 * h;
          if (r < nrows) {
            const long long g = op.idx[seg] ? (long long)__ldg(op.idx[seg] + r) : r;
            p[h] = op.base[seg] + g * op.ld[seg] - op.start[seg];
          } else {
            p[h] = nullptr;
          }
        }
      }
#pragma unroll
      for (int h = 0; h < 2; ++h)
        v[h] = p[h] ? __ldg(reinterpret_cast<const float4*>(p[h] + k0 + 4 * kq)) : make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int q = t + kGemmThreads * u;
        const int rr = q & (BM - 1), kk = q >> 7;
        const long long r = row0 + rr, k = k0 + kk;
        float val = 0.f;
        if (r < nrows && k < red_end) {
          int s = 0;
          while (k >= op.start[s + 1]) ++s;
          const long long g = op.idx[s] ? (long long)__ldg(op.idx[s] + r) : r;
          val = __ldg(op.base[s] + g * op.ld[s] + (k - op.start[s]));
        }
        sv[u] = val;
      }
    }
  }

  __device__ __forceinline__ void commit(float (*S)[LDT]) const {
    const int t = threadIdx.x;
    if constexpr (FAST) {
      const int rq = t >> 2, kq = t & 3;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        S[4 * kq + 0][rq + 64 * h] = v[h].x;
        S[4 * kq + 1][rq + 64 * h] = v[h].y;
        S[4 * kq + 2][rq + 64 * h] = v[h].z;
        S[4 * kq + 3][rq + 64 * h] = v[h].w;
      }
    } else {
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int q = t + kGemmThreads * u;
        S[q >> 7][q & (BM - 1)] = sv[u];
      }
    }
  }
};

// D operand: tile [BK reduce rows][128 cols], source is col-contiguous; staged as is
// into S[r][col].  Row gather applies to the reduce row; segments split the columns.
template <bool FAST>
struct DLoader {
  const Operand& op;
  long long col0;
  int ncols;
  int seg;       // fast: the segment this column tile lies in
  float4 v[2];
  float sv[8];

  __device__ __forceinline__ DLoader(const Operand& o, long long c0, int nc) : op(o), col0(c0), ncols(nc) {
    seg = 0;
    if constexpr (FAST) {
      while (seg + 1 < op.nseg && col0 >= op.start[seg + 1]) ++seg;
    }
  }

  __device__ __forceinline__ void fetch(long long r0, long long red_end) {
    const int t = threadIdx.x;
    if constexpr (FAST) {
      const int rr = t >> 5, c4 = t & 31;
      const long long col = col0 + 4 * c4;
      const bool col_ok = col < op.start[seg + 1] && col < ncols;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const long long r = r0 + rr + 8 * h;
        if (col_ok && r < red_end) {
          const long long g = op.idx[seg] ? (long long)__ldg(op.idx[seg] + r) : r;
          v[h] = __ldg(reinterpret_cast<const float4*>(op.base[seg] + g * op.ld[seg] + (col - op.start[seg])));
        } else {
          v[h] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    } else {
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int q = t + kGemmThreads * u;
        const int cc = q & (BN - 1), rr = q >> 7;
        const long long r = r0 + rr, c = col0 + cc;
        float val = 0.f;
        if (r < red_end && c < ncols) {
          int s = 0;
          while (c >= op.start[s + 1]) ++s;
          const long long g = op.idx[s] ? (long long)__ldg(op.idx[s] + r) : r;
          val = __ldg(op.base[s] + g * op.ld[s] + (c - op.start[s]));
        }
        sv[u] = val;
      }
    }
  }

  __device__ __forceinline__ void commit(float (*S)[LDT]) const {
    const int t = threadIdx.x;
    if constexpr (FAST) {
      const int rr = t >> 5, c4 = t & 31;
#pragma unroll
      for (int h = 0; h < 2; ++h) *reinterpret_cast<float4*>(&S[rr + 8 * h][4 * c4]) = v[h];
    } else {
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int q = t + kGemmThreads * u;
        S[q >> 7][q & (BN - 1)] = sv[u];
      }
    }
  }
};

template <bool T, bool FAST>
struct LoaderSel { using type = TLoader<FAST>; };
template <bool FAST>
struct LoaderSel<false, FAST> { using type = DLoader<FAST>; };

// EPI: 0 = forward (bias, relu), 1 = dgrad (optional accumulate), 2 = wgrad partial
template <bool A_T, bool B_T, bool FAST_A, bool FAST_B, int EPI>
__global__ void __launch_bounds__(kGemmThreads, 2) sgemm_128x128_kernel(const GemmArgs g) {
  __shared__ __align__(16) float As[2][BK][LDT];
  __shared__ __align__(16) float Bs[2][BK][LDT];

  const long long row0 = (long long)blockIdx.x * BM;
  const long long col0 = (long long)blockIdx.y * BN;
  const long long red_beg = (long long)blockIdx.z * g.red_chunk;
  long long red_end = red_beg + g.red_chunk;
  if (red_end > g.red) red_end = g.red;

  typename LoaderSel<A_T, FAST_A>::type la(g.A, row0, A_T ? g.rows : (long long)g.rows);
  typename LoaderSel<B_T, FAST_B>::type lb(g.B, col0, g.cols);
  // For a D-type A operand (wgrad) the "columns" of the source are the output rows.
  // DLoader's ctor takes (col origin, col extent): row0 / rows fit that meaning.

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tx = (warp & 1) * 8 + (lane & 7);
  const int ty = (warp >> 1) * 4 + (lane >> 3);

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  const long long ntiles = (red_end > red_beg) ? (red_end - red_beg + BK - 1) / BK : 0;
  if (ntiles > 0) {
    la.fetch(red_beg, red_end);
    lb.fetch(red_beg, red_end);
    la.commit(As[0]);
    lb.commit(Bs[0]);
  }
  __syncthreads();
  for (long long t = 0; t < ntiles; ++t) {
    const int buf = (int)(t & 1);
    const bool more = t + 1 < ntiles;
    if (more) {
      la.fetch(red_beg + (t + 1) * BK, red_end);
      lb.fetch(red_beg + (t + 1) * BK, red_end);
    }
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][kk][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][kk][64 + tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (more) {
      la.commit(As[buf ^ 1]);
      lb.commit(Bs[buf ^ 1]);
    }
    __syncthreads();
  }

  // ---- epilogue -------------------------------------------------------------
  float* C = g.C;
  if constexpr (EPI == 2) C += (long long)blockIdx.z * g.c_split_stride;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const long long r = row0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (r >= g.rows) continue;
#pragma unroll
    for (int jh = 0; jh < 2; ++jh) {
      const long long c = col0 + jh * 64 + tx * 4;
      if (c >= g.cols) continue;
      float o[4] = {acc[i][jh * 4 + 0], acc[i][jh * 4 + 1], acc[i][jh * 4 + 2], acc[i][jh * 4 + 3]};
      float* dst = C + r * g.ldc + c;
      if constexpr (EPI == 0) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (g.bias && c + j < g.cols) o[j] += __ldg(g.bias + c + j);
          if (g.relu) o[j] = fmaxf(o[j], 0.f);
        }
      }
      if (g.vec_store && c + 3 < g.cols) {
        if constexpr (EPI == 1) {
          if (g.accumulate) {
            const float4 p = *reinterpret_cast<const float4*>(dst);
            o[0] += p.x; o[1] += p.y; o[2] += p.z; o[3] += p.w;
          }
        }
        *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (c + j < g.cols) {
            if constexpr (EPI == 1) {
              if (g.accumulate) o[j] += dst[j];
            }
            dst[j] = o[j];
          }
        }
      }
    }
  }
}

// ---- host-side operand preparation ------------------------------------------
static int make_operand(const gnc_seg_t* segs, int nseg, Operand& op, long long* total) {
  if (nseg < 1 || nseg > kMaxSeg || !segs) return fail(GNC_EINVAL, "%s", "linear: need 1..3 segments");
  op.nseg = nseg;
  op.start[0] = 0;
  for (int s = 0; s < kMaxSeg; ++s) {
    if (s < nseg) {
      if (!segs[s].base || segs[s].width <= 0 || segs[s].ld < segs[s].width)
        return fail(GNC_EINVAL, "%s", "linear: bad segment (null base, width <= 0 or ld < width)");
      op.base[s] = segs[s].base; op.idx[s] = segs[s].idx; op.ld[s] = segs[s].ld;
      op.start[s + 1] = op.start[s] + segs[s].width;
    } else {
      op.base[s] = nullptr; op.idx[s] = nullptr; op.ld[s] = 0;
      op.start[s + 1] = 0x7fffffff;   // sentinel: segment searches stop here
    }
  }
  *total = op.start[nseg];
  return GNC_OK;
}

static void single_operand(const float* base, long long ld, int width, Operand& op) {
  op.nseg = 1;
  op.base[0] = base; op.idx[0] = nullptr; op.ld[0] = ld;
  op.start[0] = 0; op.start[1] = width;
  for (int s = 1; s < kMaxSeg; ++s) { op.base[s] = nullptr; op.idx[s] = nullptr; op.ld[s] = 0; op.start[s + 1] = 0x7fffffff; }
}

// T operand fast path: every segment boundary on a BK multiple, rows 16-byte aligned.
static bool t_fast(const Operand& op) {
  for (int s = 0; s < op.nseg; ++s) {
    if ((op.start[s + 1] - op.start[s]) % BK) return false;
    if (op.ld[s] % 4 || !aligned16(op.base[s])) return false;
  }
  return true;
}
// D operand fast path: column tiles never straddle segments, rows 16-byte aligned.
static bool d_fast(const Operand& op) {
  for (int s = 0; s < op.nseg; ++s) {
    const int w = op.start[s + 1] - op.start[s];
    if (op.nseg > 1 && (w % BN)) return false;
    if (w % 4 || op.ld[s] % 4 || !aligned16(op.base[s])) return false;
  }
  return true;
}

template <bool A_T, bool B_T, int EPI>
static int launch_gemm(const GemmArgs& g, bool fa, bool fb, dim3 grid, cudaStream_t st) {
  if (fa && fb) sgemm_128x128_kernel<A_T, B_T, true, true, EPI><<<grid, kGemmThreads, 0, st>>>(g);
  else if (fa) sgemm_128x128_kernel<A_T, B_T, true, false, EPI><<<grid, kGemmThreads, 0, st>>>(g);
  else if (fb) sgemm_128x128_kernel<A_T, B_T, false, true, EPI><<<grid, kGemmThreads, 0, st>>>(g);
  else sgemm_128x128_kernel<A_T, B_T, false, false, EPI><<<grid, kGemmThreads, 0, st>>>(g);
  return check_launch("sgemm_128x128_kernel");
}

static void wgrad_split(long long M, int N, int K, long long* splits, long long* chunk) {
  const long long tiles = ceil_div<long long>(N, BM) * ceil_div<long long>(K, BN);
  long long s = ceil_div<long long>(M, 1024);
  long long cap = (long long)(kNumSMs * 4) / tiles;
  if (cap < 1) cap = 1;
  if (s > cap) s = cap;
  if (s < 1) s = 1;
  long long c = ceil_div<long long>(ceil_div<long long>(M, s), BK) * BK;
  if (c < BK) c = BK;
  *chunk = c;
  *splits = M > 0 ? ceil_div<long long>(M, c) : 1;
}

__global__ void wgrad_reduce_kernel(const float* __restrict__ ws, long long splits, long long NK, int K,
                                    float* __restrict__ dW, long long lddw, int accumulate) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= NK) return;
  float s = 0.f;
  for (long long p = 0; p < splits; ++p) s += ws[p * NK + i];
  const long long n = i / K, k = i - n * K;
  float* d = dW + n * lddw + k;
  *d = accumulate ? (*d + s) : s;
}

// Split-K forward (few output tiles, long reduction: the classifier head's fc1, models/GNN.py:315): how many
// slices of the reduction run as separate CTAs, and the per-slice length.
static void fwd_split(long long M, int N, long long K, long long* splits, long long* chunk) {
  const long long tiles = ceil_div<long long>(M, BM) * ceil_div<long long>(N, BN);
  long long s = (long long)(kNumSMs * 2) / tiles;
  const long long smax = ceil_div<long long>(K, 8 * BK);      // at least 8 K-steps per slice
  if (s > smax) s = smax;
  if (s < 1) s = 1;
  long long c = ceil_div<long long>(ceil_div<long long>(K, s), BK) * BK;
  if (c < BK) c = BK;
  *chunk = c;
  *splits = ceil_div<long long>(K, c);
}

// Y[m, n] = act(sum over slices of ws[z][m, n] + bias[n]) in slice order (deterministic)
__global__ void splitk_reduce_kernel(const float* __restrict__ ws, long long splits, long long MN, int N,
                                     const float* __restrict__ bias, int relu, float* __restrict__ Y, long long ldy) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= MN) return;
  float s = 0.f;
  for (long long z = 0; z < splits; ++z) s += ws[z * MN + i];
  const long long m = i / N;
  const int n = (int)(i - m * N);
  if (bias) s += __ldg(bias + n);
  if (relu) s = fmaxf(s, 0.f);
  Y[m * ldy + n] = s;
}

// ---- column reductions --------------------------------------------------------
constexpr int kColBlocksMax = kNumSMs * 4;

static long long col_blocks(long long M) {
  long long b = ceil_div<long long>(M, 64);
  if (b > kColBlocksMax) b = kColBlocksMax;
  if (b < 1) b = 1;
  return b;
}

// dZ = dY * (Y > 0); partial[b][c] = sum over the block's rows.  Vector path: N % 4 == 0, N <= 512.
template <int VPL>
__global__ void __launch_bounds__(256) relu_bwd_colsum_vec_kernel(const float* __restrict__ dY, long long lddy,
                                                                  const float* __restrict__ Y, long long ldy,
                                                                  long long M, int N4, float* __restrict__ dZ,
                                                                  long long lddz, float* __restrict__ partial) {
  __shared__ float4 red[8][32 * VPL];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long rows_per_block = ceil_div<long long>(M, gridDim.x);
  const long long rbeg = (long long)blockIdx.x * rows_per_block;
  long long rend = rbeg + rows_per_block;
  if (rend > M) rend = M;
  float4 s[VPL];
#pragma unroll
  for (int q = 0; q < VPL; ++q) s[q] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (long long r = rbeg + warp; r < rend; r += 8) {
#pragma unroll
    for (int q = 0; q < VPL; ++q) {
      const int c4 = lane + 32 * q;
      if (c4 < N4) {
        float4 d = ldg_stream(reinterpret_cast<const float4*>(dY + r * lddy) + c4);
        if (Y) {
          const float4 y = ldg_stream(reinterpret_cast<const float4*>(Y + r * ldy) + c4);
          d.x = y.x > 0.f ? d.x : 0.f; d.y = y.y > 0.f ? d.y : 0.f;
          d.z = y.z > 0.f ? d.z : 0.f; d.w = y.w > 0.f ? d.w : 0.f;
        }
        if (dZ) *(reinterpret_cast<float4*>(dZ + r * lddz) + c4) = d;
        s[q].x += d.x; s[q].y += d.y; s[q].z += d.z; s[q].w += d.w;
      }
    }
  }
#pragma unroll
  for (int q = 0; q < VPL; ++q) red[warp][lane + 32 * q] = s[q];
  __syncthreads();
  for (int c4 = threadIdx.x; c4 < N4; c4 += blockDim.x) {
    float4 t = red[0][c4];
#pragma unroll
    for (int w = 1; w < 8; ++w) { t.x += red[w][c4].x; t.y += red[w][c4].y; t.z += red[w][c4].z; t.w += red[w][c4].w; }
    reinterpret_cast<float4*>(partial + (long long)blockIdx.x * N4 * 4)[c4] = t;
  }
}

// Any N: one thread per column inside the block's row range.
__global__ void relu_bwd_colsum_scalar_kernel(const float* __restrict__ dY, long long lddy,
                                              const float* __restrict__ Y, long long ldy, long long M, int N,
                                              float* __restrict__ dZ, long long lddz, float* __restrict__ partial) {
  const long long rows_per_block = ceil_div<long long>(M, gridDim.x);
  const long long rbeg = (long long)blockIdx.x * rows_per_block;
  long long rend = rbeg + rows_per_block;
  if (rend > M) rend = M;
  for (int c = threadIdx.x; c < N; c += blockDim.x) {
    float s = 0.f;
    for (long long r = rbeg; r < rend; ++r) {
      float d = dY[r * lddy + c];
      if (Y && !(Y[r * ldy + c] > 0.f)) d = 0.f;
      if (dZ) dZ[r * lddz + c] = d;
      s += d;
    }
    partial[(long long)blockIdx.x * N + c] = s;
  }
}

// Narrow matrices (N <= 8): the column-per-thread kernel above would leave all but
// N threads idle, so threads stride over rows instead and a block reduction follows.
__global__ void __launch_bounds__(256) relu_bwd_colsum_narrow_kernel(const float* __restrict__ dY, long long lddy,
                                                                     const float* __restrict__ Y, long long ldy,
                                                                     long long M, int N, float* __restrict__ dZ,
                                                                     long long lddz, float* __restrict__ partial) {
  __shared__ float red[256][8];
  const long long rows_per_block = ceil_div<long long>(M, gridDim.x);
  const long long rbeg = (long long)blockIdx.x * rows_per_block;
  long long rend = rbeg + rows_per_block;
  if (rend > M) rend = M;
  float s[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) s[c] = 0.f;
  for (long long r = rbeg + threadIdx.x; r < rend; r += blockDim.x) {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      if (c < N) {
        float d = dY[r * lddy + c];
        if (Y && !(Y[r * ldy + c] > 0.f)) d = 0.f;
        if (dZ) dZ[r * lddz + c] = d;
        s[c] += d;
      }
    }
  }
#pragma unroll
  for (int c = 0; c < 8; ++c) red[threadIdx.x][c] = s[c];
  __syncthreads();
  if (threadIdx.x < N) {
    float t = 0.f;
    for (int i = 0; i < 256; ++i) t += red[i][threadIdx.x];
    partial[(long long)blockIdx.x * N + threadIdx.x] = t;
  }
}

// out[c] (+)= sum_b partial[b][c]   for `nvec` stacked vectors of length N
__global__ void partial_reduce_kernel(const float* __restrict__ partial, long long blocks, int N,
                                      float* __restrict__ out, int accumulate) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= N) return;
  float s = 0.f;
  for (long long b = 0; b < blocks; ++b) s += partial[b * N + c];
  out[c] = accumulate ? out[c] + s : s;
}

// ---- Linear(D, 1) tail (the decoder's last layer, models/GNN.py:289-295 with out_channels = 1) ----------------------
// A [M, D] x [D, 1] product is a row dot product: as a GEMM it fills one column of a 128-wide tile.  Forward: one warp
// per row, 128-bit loads.  Backward (one pass over X): dX[m, :] = dy[m] * w (* (X[m, :] > 0) when X is a ReLU output
// and dX is wanted as its pre-activation gradient), dw = sum_m dy[m] X[m, :], db = sum_m dy[m].
template <int VPL>
__global__ void __launch_bounds__(256) dot_tail_fwd_kernel(const float* __restrict__ X, long long ldx, long long M, int D4,
                                                           const float* __restrict__ w, const float* __restrict__ b,
                                                           float* __restrict__ y) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float4 wv[VPL];
#pragma unroll
  for (int q = 0; q < VPL; ++q) {
    const int c4 = lane + 32 * q;
    wv[q] = c4 < D4 ? __ldg(reinterpret_cast<const float4*>(w) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const float bias = b ? __ldg(b) : 0.f;
  for (long long r = (long long)blockIdx.x * 8 + warp; r < M; r += (long long)gridDim.x * 8) {
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < VPL; ++q) {
      const int c4 = lane + 32 * q;
      if (c4 < D4) {
        const float4 x = ldg_stream(reinterpret_cast<const float4*>(X + r * ldx) + c4);
        s = fmaf(x.x, wv[q].x, s); s = fmaf(x.y, wv[q].y, s); s = fmaf(x.z, wv[q].z, s); s = fmaf(x.w, wv[q].w, s);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) y[r] = s + bias;
  }
}

template <int VPL>
__global__ void __launch_bounds__(256) dot_tail_bwd_kernel(const float* __restrict__ X, long long ldx, long long M, int D4,
                                                           const float* __restrict__ w, const float* __restrict__ dy,
                                                           int relu_mask, float* __restrict__ dX, long long lddx,
                                                           float* __restrict__ partial) {
  __shared__ float4 red[8][32 * VPL];
  __shared__ float redb[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long rows_per_block = ceil_div<long long>(M, gridDim.x);
  const long long rbeg = (long long)blockIdx.x * rows_per_block;
  long long rend = rbeg + rows_per_block;
  if (rend > M) rend = M;
  float4 wv[VPL], s[VPL];
#pragma unroll
  for (int q = 0; q < VPL; ++q) {
    const int c4 = lane + 32 * q;
    wv[q] = c4 < D4 ? __ldg(reinterpret_cast<const float4*>(w) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
    s[q] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  float sb = 0.f;
  for (long long r = rbeg + warp; r < rend; r += 8) {
    const float g = __ldg(dy + r);
    sb += g;
#pragma unroll
    for (int q = 0; q < VPL; ++q) {
      const int c4 = lane + 32 * q;
      if (c4 < D4) {
        const float4 x = ldg_stream(reinterpret_cast<const float4*>(X + r * ldx) + c4);
        s[q].x = fmaf(g, x.x, s[q].x); s[q].y = fmaf(g, x.y, s[q].y); s[q].z = fmaf(g, x.z, s[q].z); s[q].w = fmaf(g, x.w, s[q].w);
        if (dX) {
          float4 d = make_float4(g * wv[q].x, g * wv[q].y, g * wv[q].z, g * wv[q].w);
          if (relu_mask) {
            d.x = x.x > 0.f ? d.x : 0.f; d.y = x.y > 0.f ? d.y : 0.f; d.z = x.z > 0.f ? d.z : 0.f; d.w = x.w > 0.f ? d.w : 0.f;
          }
          stg_stream(reinterpret_cast<float4*>(dX + r * lddx) + c4, d);
        }
      }
    }
  }
#pragma unroll
  for (int q = 0; q < VPL; ++q) red[warp][lane + 32 * q] = s[q];
  if (lane == 0) redb[warp] = sb;
  __syncthreads();
  const int D = D4 * 4;
  for (int c4 = threadIdx.x; c4 < D4; c4 += blockDim.x) {
    float4 t = red[0][c4];
#pragma unroll
    for (int wi = 1; wi < 8; ++wi) { t.x += red[wi][c4].x; t.y += red[wi][c4].y; t.z += red[wi][c4].z; t.w += red[wi][c4].w; }
    reinterpret_cast<float4*>(partial + (long long)blockIdx.x * D)[c4] = t;
  }
  if (threadIdx.x == 0) {
    float t = 0.f;
#pragma unroll
    for (int wi = 0; wi < 8; ++wi) t += redb[wi];
    partial[(long long)gridDim.x * D + blockIdx.x] = t;
  }
}

// ---- LayerNorm ------------------------------------------------------------------
// RPW rows per warp and iteration: all of their loads (z and the residual) are issued before the first reduction, so a
// warp keeps RPW x 1 KB in flight instead of 512 B (one row per iteration left the kernel latency-bound at ~60 % of HBM).
template <int VPL, int RPW>
__global__ void __launch_bounds__(256) layernorm_fwd_vec_kernel(const float* __restrict__ z, long long ldz,
                                                                long long M, int D, const float* __restrict__ gamma,
                                                                const float* __restrict__ beta, float eps,
                                                                const float* __restrict__ res, long long ldres,
                                                                float* __restrict__ y, long long ldy,
                                                                float* __restrict__ mean, float* __restrict__ rstd) {
  const int lane = threadIdx.x & 31;
  const int D4 = D >> 2;
  const long long warp_global = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long warps_total = ((long long)gridDim.x * blockDim.x) >> 5;
  float4 g[VPL], bt[VPL];
#pragma unroll
  for (int q = 0; q < VPL; ++q) {
    const int c4 = lane + 32 * q;
    g[q] = (c4 < D4) ? __ldg(reinterpret_cast<const float4*>(gamma) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
    bt[q] = (c4 < D4) ? __ldg(reinterpret_cast<const float4*>(beta) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (long long r0 = warp_global * RPW; r0 < M; r0 += warps_total * RPW) {
    float4 v[RPW][VPL], p[RPW][VPL];
#pragma unroll
    for (int t = 0; t < RPW; ++t) {
      const long long r = r0 + t;
#pragma unroll
      for (int q = 0; q < VPL; ++q) {
        const int c4 = lane + 32 * q;
        const bool ok = r < M && c4 < D4;
        v[t][q] = ok ? ldg_stream(reinterpret_cast<const float4*>(z + r * ldz) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
        p[t][q] = (ok && res) ? ldg_stream(reinterpret_cast<const float4*>(res + r * ldres) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
#pragma unroll
    for (int t = 0; t < RPW; ++t) {
      const long long r = r0 + t;
      if (r >= M) break;
      float s = 0.f;
#pragma unroll
      for (int q = 0; q < VPL; ++q) s += (v[t][q].x + v[t][q].y) + (v[t][q].z + v[t][q].w);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      const float mu = s / (float)D;      // (a division: exact for a constant row whatever D)
      float ss = 0.f;
#pragma unroll
      for (int q = 0; q < VPL; ++q) {
        const int c4 = lane + 32 * q;
        if (c4 < D4) {
          const float a = v[t][q].x - mu, b = v[t][q].y - mu, c = v[t][q].z - mu, d = v[t][q].w - mu;
          ss += (a * a + b * b) + (c * c + d * d);
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
      const float rs = 1.0f / sqrtf(ss / (float)D + eps);
      if (lane == 0) {
        if (mean) mean[r] = mu;
        if (rstd) rstd[r] = rs;
      }
#pragma unroll
      for (int q = 0; q < VPL; ++q) {
        const int c4 = lane + 32 * q;
        if (c4 < D4) {
          float4 o;
          o.x = (v[t][q].x - mu) * rs * g[q].x + bt[q].x;
          o.y = (v[t][q].y - mu) * rs * g[q].y + bt[q].y;
          o.z = (v[t][q].z - mu) * rs * g[q].z + bt[q].z;
          o.w = (v[t][q].w - mu) * rs * g[q].w + bt[q].w;
          if (res) { o.x += p[t][q].x; o.y += p[t][q].y; o.z += p[t][q].z; o.w += p[t][q].w; }
          stg_stream(reinterpret_cast<float4*>(y + r * ldy) + c4, o);
        }
      }
    }
  }
}

__global__ void __launch_bounds__(256) layernorm_fwd_scalar_kernel(const float* __restrict__ z, long long ldz,
                                                                   long long M, int D, const float* __restrict__ gamma,
                                                                   const float* __restrict__ beta, float eps,
                                                                   const float* __restrict__ res, long long ldres,
                                                                   float* __restrict__ y, long long ldy,
                                                                   float* __restrict__ mean, float* __restrict__ rstd) {
  const int lane = threadIdx.x & 31;
  const long long warp_global = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long warps_total = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r = warp_global; r < M; r += warps_total) {
    const float* zr = z + r * ldz;
    float s = 0.f;
    for (int c = lane; c < D; c += 32) s += zr[c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    float mu = s / (float)D;
    // corrected two-pass: the deviations from the first mean also sum to D times its rounding error, which matters when
    // the row's centre is far from zero against its spread
    float sd = 0.f, ss = 0.f;
    for (int c = lane; c < D; c += 32) { const float a = zr[c] - mu; sd += a; ss += a * a; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      sd += __shfl_xor_sync(0xffffffffu, sd, o);
      ss += __shfl_xor_sync(0xffffffffu, ss, o);
    }
    const float dm = sd / (float)D;
    mu += dm;
    const float rs = 1.0f / sqrtf(fmaxf(ss / (float)D - dm * dm, 0.f) + eps);
    if (lane == 0) {
      if (mean) mean[r] = mu;
      if (rstd) rstd[r] = rs;
    }
    for (int c = lane; c < D; c += 32) {
      float o = (zr[c] - mu) * rs * gamma[c] + beta[c];
      if (res) o += res[r * ldres + c];
      y[r * ldy + c] = o;
    }
  }
}

// dz = rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dy * gamma
// partial[b][0][c] = sum dy * xhat, partial[b][1][c] = sum dy  over the block's rows
template <int VPL, int RPW>
__global__ void __launch_bounds__(256) layernorm_bwd_vec_kernel(const float* __restrict__ dy, long long lddy,
                                                                const float* __restrict__ z, long long ldz,
                                                                const float* __restrict__ mean,
                                                                const float* __restrict__ rstd,
                                                                const float* __restrict__ gamma, long long M, int D,
                                                                float* __restrict__ dz, long long lddz,
                                                                float* __restrict__ partial) {
  __shared__ float4 red[8][2][32 * VPL];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int D4 = D >> 2;
  const float invD = 1.0f / (float)D;
  const long long rows_per_block = ceil_div<long long>(M, gridDim.x);
  const long long rbeg = (long long)blockIdx.x * rows_per_block;
  long long rend = rbeg + rows_per_block;
  if (rend > M) rend = M;
  float4 gm[VPL], sg[VPL], sb[VPL];
#pragma unroll
  for (int q = 0; q < VPL; ++q) {
    const int c4 = lane + 32 * q;
    gm[q] = (c4 < D4) ? __ldg(reinterpret_cast<const float4*>(gamma) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
    sg[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    sb[q] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (long long r0 = rbeg + warp; r0 < rend; r0 += 8 * RPW) {
    // RPW rows of this warp (r0, r0 + 8, ...) with all loads issued up front; rows are retired in the same order as
    // a one-row-per-iteration loop, so the column sums are bit-identical to it
    float4 d[RPW][VPL], zz[RPW][VPL];
    float mu[RPW], rs[RPW];
#pragma unroll
    for (int t = 0; t < RPW; ++t) {
      const long long r = r0 + 8 * t;
      const bool okr = r < rend;
      mu[t] = okr ? __ldg(mean + r) : 0.f;
      rs[t] = okr ? __ldg(rstd + r) : 0.f;
#pragma unroll
      for (int q = 0; q < VPL; ++q) {
        const int c4 = lane + 32 * q;
        const bool ok = okr && c4 < D4;
        d[t][q] = ok ? ldg_stream(reinterpret_cast<const float4*>(dy + r * lddy) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
        zz[t][q] = ok ? ldg_stream(reinterpret_cast<const float4*>(z + r * ldz) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
#pragma unroll
    for (int t = 0; t < RPW; ++t) {
      const long long r = r0 + 8 * t;
      if (r >= rend) break;
      float4 xh[VPL];
      float c1 = 0.f, c2 = 0.f;
#pragma unroll
      for (int q = 0; q < VPL; ++q) {
        const int c4 = lane + 32 * q;
        if (c4 < D4) {
          xh[q] = make_float4((zz[t][q].x - mu[t]) * rs[t], (zz[t][q].y - mu[t]) * rs[t], (zz[t][q].z - mu[t]) * rs[t],
                              (zz[t][q].w - mu[t]) * rs[t]);
        } else {
          xh[q] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        const float4 dd = d[t][q];
        sg[q].x += dd.x * xh[q].x; sg[q].y += dd.y * xh[q].y; sg[q].z += dd.z * xh[q].z; sg[q].w += dd.w * xh[q].w;
        sb[q].x += dd.x; sb[q].y += dd.y; sb[q].z += dd.z; sb[q].w += dd.w;
        const float gx = dd.x * gm[q].x, gy = dd.y * gm[q].y, gz = dd.z * gm[q].z, gw = dd.w * gm[q].w;
        c1 += (gx + gy) + (gz + gw);
        c2 += (gx * xh[q].x + gy * xh[q].y) + (gz * xh[q].z + gw * xh[q].w);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        c1 += __shfl_xor_sync(0xffffffffu, c1, o);
        c2 += __shfl_xor_sync(0xffffffffu, c2, o);
      }
      c1 *= invD; c2 *= invD;
#pragma unroll
      for (int q = 0; q < VPL; ++q) {
        const int c4 = lane + 32 * q;
        if (c4 < D4) {
          const float4 dd = d[t][q];
          float4 o;
          o.x = rs[t] * (dd.x * gm[q].x - c1 - xh[q].x * c2);
          o.y = rs[t] * (dd.y * gm[q].y - c1 - xh[q].y * c2);
          o.z = rs[t] * (dd.z * gm[q].z - c1 - xh[q].z * c2);
          o.w = rs[t] * (dd.w * gm[q].w - c1 - xh[q].w * c2);
          stg_stream(reinterpret_cast<float4*>(dz + r * lddz) + c4, o);
        }
      }
    }
  }
#pragma unroll
  for (int q = 0; q < VPL; ++q) { red[warp][0][lane + 32 * q] = sg[q]; red[warp][1][lane + 32 * q] = sb[q]; }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * D4; i += blockDim.x) {
    const int which = i / D4, c4 = i - which * D4;
    float4 t = red[0][which][c4];
#pragma unroll
    for (int w = 1; w < 8; ++w) {
      const float4 u = red[w][which][c4];
      t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w;
    }
    reinterpret_cast<float4*>(partial + ((long long)blockIdx.x * 2 + which) * D)[c4] = t;
  }
}

// Any D: one warp per row for dz; column partials with one thread per column afterwards.
__global__ void __launch_bounds__(256) layernorm_bwd_scalar_kernel(const float* __restrict__ dy, long long lddy,
                                                                   const float* __restrict__ z, long long ldz,
                                                                   const float* __restrict__ mean,
                                                                   const float* __restrict__ rstd,
                                                                   const float* __restrict__ gamma, long long M, int D,
                                                                   float* __restrict__ dz, long long lddz,
                                                                   float* __restrict__ partial) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float invD = 1.0f / (float)D;
  const long long rows_per_block = ceil_div<long long>(M, gridDim.x);
  const long long rbeg = (long long)blockIdx.x * rows_per_block;
  long long rend = rbeg + rows_per_block;
  if (rend > M) rend = M;
  for (long long r = rbeg + warp; r < rend; r += 8) {
    const float mu = mean[r], rs = rstd[r];
    float c1 = 0.f, c2 = 0.f;
    for (int c = lane; c < D; c += 32) {
      const float g = dy[r * lddy + c] * gamma[c];
      c1 += g;
      c2 += g * ((z[r * ldz + c] - mu) * rs);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      c1 += __shfl_xor_sync(0xffffffffu, c1, o);
      c2 += __shfl_xor_sync(0xffffffffu, c2, o);
    }
    c1 *= invD; c2 *= invD;
    for (int c = lane; c < D; c += 32) {
      const float xh = (z[r * ldz + c] - mu) * rs;
      dz[r * lddz + c] = rs * (dy[r * lddy + c] * gamma[c] - c1 - xh * c2);
    }
  }
  for (int c = threadIdx.x; c < D; c += blockDim.x) {
    float sg = 0.f, sb = 0.f;
    for (long long r = rbeg; r < rend; ++r) {
      const float d = dy[r * lddy + c];
      sg += d * ((z[r * ldz + c] - mean[r]) * rstd[r]);
      sb += d;
    }
    partial[((long long)blockIdx.x * 2 + 0) * D + c] = sg;
    partial[((long long)blockIdx.x * 2 + 1) * D + c] = sb;
  }
}

// partial [blocks][2][D] -> dgamma, dbeta
__global__ void layernorm_param_reduce_kernel(const float* __restrict__ partial, long long blocks, int D,
                                              float* __restrict__ dgamma, float* __restrict__ dbeta, int accumulate) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 2 * D) return;
  const int which = i / D, c = i - which * D;
  float s = 0.f;
  for (long long b = 0; b < blocks; ++b) s += partial[(b * 2 + which) * D + c];
  float* out = which == 0 ? dgamma : dbeta;
  if (out) out[c] = accumulate ? out[c] + s : s;
}

}  // namespace gnc

using namespace gnc;

extern "C" {

int gnc_linear_fwd_f32(const gnc_seg_t* segs, int nseg, int64_t M, const float* W, int64_t ldw, const float* bias,
                       int N, int relu, float* Y, int64_t ldy, gnc_stream_t stream) {
  GNC_REQUIRE(M >= 0 && N > 0 && W && Y && ldy >= N, "linear_fwd: bad arguments");
  if (M == 0) return GNC_OK;
  GemmArgs g;
  long long K = 0;
  int rc = make_operand(segs, nseg, g.A, &K);
  if (rc) return rc;
  GNC_REQUIRE(ldw >= K, "linear_fwd: ldw < K");
  single_operand(W, ldw, (int)K, g.B);
  g.rows = M; g.cols = N; g.red = K; g.red_chunk = ceil_div<long long>(K, BK) * BK;
  g.C = Y; g.ldc = ldy; g.c_split_stride = 0; g.bias = bias; g.relu = relu; g.accumulate = 0;
  g.vec_store = (ldy % 4 == 0 && aligned16(Y)) ? 1 : 0;
  dim3 grid((unsigned)ceil_div<long long>(M, BM), (unsigned)ceil_div<long long>(N, BN), 1);
  return launch_gemm<true, true, 0>(g, t_fast(g.A), t_fast(g.B), grid, (cudaStream_t)stream);
}

int64_t gnc_linear_fwd_splitk_workspace(int64_t M, int N, int64_t K) {
  long long splits, chunk;
  fwd_split(M, N, K, &splits, &chunk);
  return splits > 1 ? splits * M * (int64_t)N : 0;
}

int gnc_linear_fwd_splitk_f32(const gnc_seg_t* segs, int nseg, int64_t M, const float* W, int64_t ldw, const float* bias,
                              int N, int relu, float* Y, int64_t ldy, float* work, int64_t work_elems,
                              gnc_stream_t stream) {
  GNC_REQUIRE(M >= 0 && N > 0 && W && Y && ldy >= N, "linear_fwd_splitk: bad arguments");
  if (M == 0) return GNC_OK;
  GemmArgs g;
  long long K = 0;
  int rc = make_operand(segs, nseg, g.A, &K);
  if (rc) return rc;
  GNC_REQUIRE(ldw >= K, "linear_fwd_splitk: ldw < K");
  long long splits, chunk;
  fwd_split(M, N, K, &splits, &chunk);
  if (splits <= 1) return gnc_linear_fwd_f32(segs, nseg, M, W, ldw, bias, N, relu, Y, ldy, stream);
  const long long MN = (long long)M * N;
  if (!work || work_elems < splits * MN) return fail(GNC_EWORKSPACE, "%s", "linear_fwd_splitk: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  single_operand(W, ldw, (int)K, g.B);
  g.rows = M; g.cols = N; g.red = K; g.red_chunk = chunk;
  g.C = work; g.ldc = N; g.c_split_stride = MN; g.bias = nullptr; g.relu = 0; g.accumulate = 0;
  g.vec_store = (N % 4 == 0 && aligned16(work)) ? 1 : 0;
  dim3 grid((unsigned)ceil_div<long long>(M, BM), (unsigned)ceil_div<long long>(N, BN), (unsigned)splits);
  rc = launch_gemm<true, true, 2>(g, t_fast(g.A), t_fast(g.B), grid, st);
  if (rc) return rc;
  splitk_reduce_kernel<<<(unsigned)ceil_div<long long>(MN, 256), 256, 0, st>>>(work, splits, MN, N, bias, relu, Y, ldy);
  return check_launch("splitk_reduce_kernel");
}

int gnc_linear_dgrad_f32(const float* dZ, int64_t lddz, int64_t M, int N, const float* W, int64_t ldw, int K,
                         float* dX, int64_t lddx, int accumulate, gnc_stream_t stream) {
  GNC_REQUIRE(M >= 0 && N > 0 && K > 0 && dZ && W && dX && lddz >= N && ldw >= K && lddx >= K,
              "linear_dgrad: bad arguments");
  if (M == 0) return GNC_OK;
  GemmArgs g;
  single_operand(dZ, lddz, N, g.A);
  single_operand(W, ldw, K, g.B);
  g.rows = M; g.cols = K; g.red = N; g.red_chunk = ceil_div<long long>(N, BK) * BK;
  g.C = dX; g.ldc = lddx; g.c_split_stride = 0; g.bias = nullptr; g.relu = 0; g.accumulate = accumulate;
  g.vec_store = (lddx % 4 == 0 && aligned16(dX)) ? 1 : 0;
  dim3 grid((unsigned)ceil_div<long long>(M, BM), (unsigned)ceil_div<long long>(K, BN), 1);
  return launch_gemm<true, false, 1>(g, t_fast(g.A), d_fast(g.B), grid, (cudaStream_t)stream);
}

int64_t gnc_linear_wgrad_workspace(int64_t M, int N, int K) {
  long long splits, chunk;
  wgrad_split(M, N, K, &splits, &chunk);
  return splits * (int64_t)N * K;
}

int gnc_linear_wgrad_f32(const float* dZ, int64_t lddz, int64_t M, int N, const gnc_seg_t* segs, int nseg,
                         float* dW, int64_t lddw, int accumulate, float* work, int64_t work_elems,
                         gnc_stream_t stream) {
  GNC_REQUIRE(M >= 0 && N > 0 && dZ && dW && lddz >= N, "linear_wgrad: bad arguments");
  GemmArgs g;
  long long K = 0;
  int rc = make_operand(segs, nseg, g.B, &K);
  if (rc) return rc;
  GNC_REQUIRE(lddw >= K, "linear_wgrad: lddw < K");
  long long splits, chunk;
  wgrad_split(M, N, (int)K, &splits, &chunk);
  if (!work || work_elems < splits * (long long)N * K) return fail(GNC_EWORKSPACE, "%s", "linear_wgrad: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  if (M > 0) {
    single_operand(dZ, lddz, N, g.A);
    g.rows = N; g.cols = (int)K; g.red = M; g.red_chunk = chunk;
    g.C = work; g.ldc = K; g.c_split_stride = (long long)N * K; g.bias = nullptr; g.relu = 0; g.accumulate = 0;
    g.vec_store = (K % 4 == 0 && aligned16(work)) ? 1 : 0;
    dim3 grid((unsigned)ceil_div<long long>(N, BM), (unsigned)ceil_div<long long>(K, BN), (unsigned)splits);
    rc = launch_gemm<false, false, 2>(g, d_fast(g.A), d_fast(g.B), grid, st);
    if (rc) return rc;
  } else {
    splits = 0;
  }
  const long long NK = (long long)N * K;
  wgrad_reduce_kernel<<<(unsigned)ceil_div<long long>(NK, 256), 256, 0, st>>>(work, splits, NK, (int)K, dW, lddw,
                                                                             accumulate);
  return check_launch("wgrad_reduce_kernel");
}

int gnc_dot_tail_fwd_f32(const float* X, int64_t ldx, int64_t M, int D, const float* w, const float* b, float* y,
                         gnc_stream_t stream) {
  GNC_REQUIRE(X && w && y && M >= 0 && D > 0 && D % 4 == 0 && D <= 512 && ldx >= D && ldx % 4 == 0 && aligned16(X) && aligned16(w),
              "dot_tail_fwd: D % 4 == 0, D <= 512, 16-byte aligned rows");
  if (M == 0) return GNC_OK;
  cudaStream_t st = (cudaStream_t)stream;
  long long blocks = ceil_div<long long>(M, 8);
  if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
  const int D4 = D / 4;
  if (D4 <= 32) dot_tail_fwd_kernel<1><<<(unsigned)blocks, 256, 0, st>>>(X, ldx, M, D4, w, b, y);
  else if (D4 <= 64) dot_tail_fwd_kernel<2><<<(unsigned)blocks, 256, 0, st>>>(X, ldx, M, D4, w, b, y);
  else dot_tail_fwd_kernel<4><<<(unsigned)blocks, 256, 0, st>>>(X, ldx, M, D4, w, b, y);
  return check_launch("dot_tail_fwd_kernel");
}

int64_t gnc_dot_tail_bwd_workspace(int64_t M, int D) { return col_blocks(M) * (int64_t)(D + 1); }

int gnc_dot_tail_bwd_f32(const float* X, int64_t ldx, int64_t M, int D, const float* w, const float* dy, int relu_mask,
                         float* dX, int64_t lddx, float* dw, float* db, int accumulate, float* work, int64_t work_elems,
                         gnc_stream_t stream) {
  GNC_REQUIRE(X && w && dy && M >= 0 && D > 0 && D % 4 == 0 && D <= 512 && ldx >= D && ldx % 4 == 0 && aligned16(X) && aligned16(w),
              "dot_tail_bwd: D % 4 == 0, D <= 512, 16-byte aligned rows");
  GNC_REQUIRE(!dX || (lddx >= D && lddx % 4 == 0 && aligned16(dX)), "dot_tail_bwd: dX rows must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const long long blocks = col_blocks(M);
  if (!work || work_elems < blocks * (long long)(D + 1)) return fail(GNC_EWORKSPACE, "%s", "dot_tail_bwd: workspace too small");
  const int D4 = D / 4;
  if (D4 <= 32) dot_tail_bwd_kernel<1><<<(unsigned)blocks, 256, 0, st>>>(X, ldx, M, D4, w, dy, relu_mask, dX, lddx, work);
  else if (D4 <= 64) dot_tail_bwd_kernel<2><<<(unsigned)blocks, 256, 0, st>>>(X, ldx, M, D4, w, dy, relu_mask, dX, lddx, work);
  else dot_tail_bwd_kernel<4><<<(unsigned)blocks, 256, 0, st>>>(X, ldx, M, D4, w, dy, relu_mask, dX, lddx, work);
  int rc = check_launch("dot_tail_bwd_kernel");
  if (rc) return rc;
  if (dw) {
    partial_reduce_kernel<<<(unsigned)ceil_div<int>(D, 256), 256, 0, st>>>(work, blocks, D, dw, accumulate);
    if ((rc = check_launch("partial_reduce_kernel"))) return rc;
  }
  if (db) {
    // the per-block scalars are a [blocks][1] stack: same fixed-order reduction with N = 1
    partial_reduce_kernel<<<1, 32, 0, st>>>(work + blocks * (long long)D, blocks, 1, db, accumulate);
    if ((rc = check_launch("partial_reduce_kernel"))) return rc;
  }
  return GNC_OK;
}

int64_t gnc_colsum_workspace(int64_t M, int N) { return col_blocks(M) * (int64_t)N; }

int gnc_relu_bwd_colsum_f32(const float* dY, int64_t lddy, const float* Y, int64_t ldy, int64_t M, int N, float* dZ,
                            int64_t lddz, float* db, int accumulate, float* work, int64_t work_elems,
                            gnc_stream_t stream) {
  GNC_REQUIRE(M >= 0 && N > 0 && dY && lddy >= N, "relu_bwd_colsum: bad arguments");
  GNC_REQUIRE(!Y || ldy >= N, "relu_bwd_colsum: ldy < N");
  GNC_REQUIRE(!dZ || lddz >= N, "relu_bwd_colsum: lddz < N");
  cudaStream_t st = (cudaStream_t)stream;
  const long long blocks = M > 0 ? col_blocks(M) : 0;
  if (!work || work_elems < blocks * (long long)N) return fail(GNC_EWORKSPACE, "%s", "relu_bwd_colsum: workspace too small");
  int rc;
  if (M > 0) {
    const bool vec = N % 4 == 0 && N <= 512 && lddy % 4 == 0 && aligned16(dY) && (!Y || (ldy % 4 == 0 && aligned16(Y))) &&
                     (!dZ || (lddz % 4 == 0 && aligned16(dZ))) && aligned16(work);
    if (vec) {
      const int N4 = N / 4;
      if (N4 <= 32) relu_bwd_colsum_vec_kernel<1><<<(unsigned)blocks, 256, 0, st>>>(dY, lddy, Y, ldy, M, N4, dZ, lddz, work);
      else if (N4 <= 64) relu_bwd_colsum_vec_kernel<2><<<(unsigned)blocks, 256, 0, st>>>(dY, lddy, Y, ldy, M, N4, dZ, lddz, work);
      else relu_bwd_colsum_vec_kernel<4><<<(unsigned)blocks, 256, 0, st>>>(dY, lddy, Y, ldy, M, N4, dZ, lddz, work);
    } else if (N <= 8) {
      relu_bwd_colsum_narrow_kernel<<<(unsigned)blocks, 256, 0, st>>>(dY, lddy, Y, ldy, M, N, dZ, lddz, work);
    } else {
      relu_bwd_colsum_scalar_kernel<<<(unsigned)blocks, 256, 0, st>>>(dY, lddy, Y, ldy, M, N, dZ, lddz, work);
    }
    if ((rc = check_launch("relu_bwd_colsum_kernel"))) return rc;
  }
  if (db) {
    partial_reduce_kernel<<<(unsigned)ceil_div<int>(N, 256), 256, 0, st>>>(work, blocks, N, db, accumulate);
    if ((rc = check_launch("partial_reduce_kernel"))) return rc;
  }
  return GNC_OK;
}

int gnc_layernorm_fwd_f32(const float* z, int64_t ldz, int64_t M, int D, const float* gamma, const float* beta,
                          float eps, const float* res, int64_t ldres, float* y, int64_t ldy, float* mean, float* rstd,
                          gnc_stream_t stream) {
  GNC_REQUIRE(M >= 0 && D > 0 && z && gamma && beta && y && ldz >= D && ldy >= D, "layernorm_fwd: bad arguments");
  GNC_REQUIRE(!res || ldres >= D, "layernorm_fwd: ldres < D");
  if (M == 0) return GNC_OK;
  cudaStream_t st = (cudaStream_t)stream;
  long long blocks = ceil_div<long long>(M, 8);
  if (blocks > (long long)kNumSMs * 8) blocks = (long long)kNumSMs * 8;
  const bool vec = D % 4 == 0 && D <= 512 && ldz % 4 == 0 && ldy % 4 == 0 && aligned16(z) && aligned16(y) &&
                   aligned16(gamma) && aligned16(beta) && (!res || (ldres % 4 == 0 && aligned16(res)));
  if (vec) {
    const int D4 = D / 4;
    if (D4 <= 32) layernorm_fwd_vec_kernel<1, 4><<<(unsigned)blocks, 256, 0, st>>>(z, ldz, M, D, gamma, beta, eps, res, ldres, y, ldy, mean, rstd);
    else if (D4 <= 64) layernorm_fwd_vec_kernel<2, 2><<<(unsigned)blocks, 256, 0, st>>>(z, ldz, M, D, gamma, beta, eps, res, ldres, y, ldy, mean, rstd);
    else layernorm_fwd_vec_kernel<4, 1><<<(unsigned)blocks, 256, 0, st>>>(z, ldz, M, D, gamma, beta, eps, res, ldres, y, ldy, mean, rstd);
  } else {
    layernorm_fwd_scalar_kernel<<<(unsigned)blocks, 256, 0, st>>>(z, ldz, M, D, gamma, beta, eps, res, ldres, y, ldy, mean, rstd);
  }
  return check_launch("layernorm_fwd_kernel");
}

int64_t gnc_layernorm_bwd_workspace(int64_t M, int D) { return col_blocks(M) * 2 * (int64_t)D; }

int gnc_layernorm_bwd_f32(const float* dy, int64_t lddy, const float* z, int64_t ldz, const float* mean,
                          const float* rstd, const float* gamma, int64_t M, int D, float* dz, int64_t lddz,
                          float* dgamma, float* dbeta, int accumulate, float* work, int64_t work_elems,
                          gnc_stream_t stream) {
  GNC_REQUIRE(M >= 0 && D > 0 && dy && z && mean && rstd && gamma && dz && lddy >= D && ldz >= D && lddz >= D,
              "layernorm_bwd: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const long long blocks = M > 0 ? col_blocks(M) : 0;
  if (!work || work_elems < blocks * 2 * (long long)D) return fail(GNC_EWORKSPACE, "%s", "layernorm_bwd: workspace too small");
  int rc;
  if (M > 0) {
    const bool vec = D % 4 == 0 && D <= 512 && lddy % 4 == 0 && ldz % 4 == 0 && lddz % 4 == 0 && aligned16(dy) &&
                     aligned16(z) && aligned16(dz) && aligned16(gamma) && aligned16(work);
    if (vec) {
      const int D4 = D / 4;
      if (D4 <= 32) layernorm_bwd_vec_kernel<1, 4><<<(unsigned)blocks, 256, 0, st>>>(dy, lddy, z, ldz, mean, rstd, gamma, M, D, dz, lddz, work);
      else if (D4 <= 64) layernorm_bwd_vec_kernel<2, 2><<<(unsigned)blocks, 256, 0, st>>>(dy, lddy, z, ldz, mean, rstd, gamma, M, D, dz, lddz, work);
      else layernorm_bwd_vec_kernel<4, 1><<<(unsigned)blocks, 256, 0, st>>>(dy, lddy, z, ldz, mean, rstd, gamma, M, D, dz, lddz, work);
    } else {
      layernorm_bwd_scalar_kernel<<<(unsigned)blocks, 256, 0, st>>>(dy, lddy, z, ldz, mean, rstd, gamma, M, D, dz, lddz, work);
    }
    if ((rc = check_launch("layernorm_bwd_kernel"))) return rc;
  }
  if (dgamma || dbeta) {
    layernorm_param_reduce_kernel<<<(unsigned)ceil_div<int>(2 * D, 256), 256, 0, st>>>(work, blocks, D, dgamma, dbeta, accumulate);
    if ((rc = check_launch("layernorm_param_reduce_kernel"))) return rc;
  }
  return GNC_OK;
}

}  // extern "C"
