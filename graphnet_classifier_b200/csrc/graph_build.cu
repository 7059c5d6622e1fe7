// Graph construction kernels (sm_100a): batched pixel / patch grid graphs emitted
// directly with their CSR, generic stable CSR from an arbitrary edge_index, and the
// label-map -> superpixel-graph stage.  All HBM-bound integer/byte work: one pass,
// coalesced 128-bit stores, grids sized in multiples of the SM count.
//
// Reference behaviour restated (paths relative to the reference root):
//   utils/image_to_graph/image_to_graph_optimized.py:7-39, 71-87
//   utils/image_to_graph/image_to_graph_patch.py:25-54
//   utils/image_to_graph/image_to_graph_superpixel.py:34-71
//   utils/dataloader.py:49-51 (casts to float32 / float32 / int64)
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"
#include "grid_topology.h"

namespace gnc {

thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};

// ----------------------------------------------------------------------------
// Fused grid-graph builder.  One launch covers four item ranges ("phases"):
//   A  node features   (pixel: 16 image bytes -> 16 floats per item;
//                       patch: one tile mean per item)
//   B  node positions  (one node per item, float2 store)
//   C  edge list       (one edge per item: int64 src/dst rows + int32 copies)
//   D  CSR by dst and by src (one node per item, closed form - no sort)
// ----------------------------------------------------------------------------
struct GridBuildArgs {
  const uint8_t* img;
  float* x;
  float* pos;
  int64_t* ei;
  int32_t *src32, *dst32, *drp, *deid, *srp, *seid;
  int B, imgH, imgW, patch;   // patch == 0: pixel graph
  GridDims g;                 // node grid (pixels or tiles)
  int64_t endA, endB, endC, endD;
  int vecA;                   // phase A uses 16-byte items
};

__device__ __forceinline__ void phase_pixel_features(const GridBuildArgs& a, int64_t it) {
  const int64_t nbytes = (int64_t)a.B * a.g.N * 3;
  if (a.vecA) {
    // unit `it` = 16 input bytes, but the 32 units of a warp are walked word-interleaved: lane l takes the
    // 32-bit words l, l + 32, l + 64, l + 96 of the warp's 512-byte block, so that every load is one coalesced
    // 128-byte request and every store one coalesced 512-byte request (4 pixels' channels per float4)
    const int64_t wbase = (it & ~(int64_t)31) * 4 + (it & 31);      // first word of this lane
    const int64_t nwords = nbytes >> 2;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int64_t w = wbase + 32 * k;
      if (w < nwords) {
        const uint32_t q = __ldg(reinterpret_cast<const uint32_t*>(a.img) + w);
        float4 f;
        f.x = (float)(q & 0xffu);
        f.y = (float)((q >> 8) & 0xffu);
        f.z = (float)((q >> 16) & 0xffu);
        f.w = (float)(q >> 24);
        stg_stream(reinterpret_cast<float4*>(a.x) + w, f);
      } else if (w == nwords) {
        for (int64_t p = nwords * 4; p < nbytes; ++p) a.x[p] = (float)a.img[p];   // < 4 trailing bytes
      }
    }
  } else {
    const int64_t off = it * 16;
    const int64_t end = off + 16 < nbytes ? off + 16 : nbytes;
    for (int64_t p = off; p < end; ++p) a.x[p] = (float)a.img[p];
  }
}

// np.mean over a p x p uint8 tile: exact integer sum, one float64 division, then
// the loader's float32 cast (image_to_graph_patch.py:40-41, dataloader.py:49).
__device__ __forceinline__ void phase_patch_features(const GridBuildArgs& a, int64_t gv) {
  const int64_t b = gv / a.g.N, v = gv - b * a.g.N;
  const int ti = (int)(v / a.g.W), tj = (int)(v - (int64_t)ti * a.g.W);
  const int p = a.patch;
  const uint8_t* base = a.img + ((b * a.imgH + (int64_t)ti * p) * a.imgW + (int64_t)tj * p) * 3;
  uint32_t s0 = 0, s1 = 0, s2 = 0;
  for (int r = 0; r < p; ++r) {
    const uint8_t* row = base + (int64_t)r * a.imgW * 3;
    for (int c = 0; c < p; ++c) {
      s0 += row[3 * c]; s1 += row[3 * c + 1]; s2 += row[3 * c + 2];
    }
  }
  const double inv = (double)(p * p);
  a.x[gv * 3 + 0] = (float)((double)s0 / inv);
  a.x[gv * 3 + 1] = (float)((double)s1 / inv);
  a.x[gv * 3 + 2] = (float)((double)s2 / inv);
}

__device__ __forceinline__ void phase_positions(const GridBuildArgs& a, int64_t gv) {
  const int64_t v = gv % a.g.N;
  const int i = (int)(v / a.g.W), j = (int)(v - (int64_t)i * a.g.W);
  float2 p;
  if (a.patch) {
    p.x = (float)(i * a.patch + a.patch / 2);
    p.y = (float)(j * a.patch + a.patch / 2);
  } else {
    p.x = (float)i; p.y = (float)j;
  }
  reinterpret_cast<float2*>(a.pos)[gv] = p;
}

__device__ __forceinline__ void phase_edges(const GridBuildArgs& a, int64_t ge) {
  const int64_t b = ge / a.g.E, e = ge - b * a.g.E;
  int64_t s, d;
  grid_edge(a.g, e, s, d);
  s += b * a.g.N; d += b * a.g.N;
  if (a.ei) {
    const int64_t BE = (int64_t)a.B * a.g.E;
    a.ei[ge] = s;
    a.ei[BE + ge] = d;
  }
  if (a.src32) { a.src32[ge] = (int32_t)s; a.dst32[ge] = (int32_t)d; }
}

__device__ __forceinline__ void phase_csr(const GridBuildArgs& a, int64_t gv) {
  const int64_t b = gv / a.g.N, v = gv - b * a.g.N;
  const int64_t eoff = b * a.g.E;
  int64_t ids[4], before;
  int n = grid_in_edges(a.g, v, ids, &before);
  a.drp[gv] = (int32_t)(eoff + before);
  for (int k = 0; k < n; ++k) a.deid[eoff + before + k] = (int32_t)(eoff + ids[k]);
  n = grid_out_edges(a.g, v, ids, &before);
  a.srp[gv] = (int32_t)(eoff + before);
  for (int k = 0; k < n; ++k) a.seid[eoff + before + k] = (int32_t)(eoff + ids[k]);
  if (gv == (int64_t)a.B * a.g.N - 1) {
    a.drp[gv + 1] = (int32_t)((int64_t)a.B * a.g.E);
    a.srp[gv + 1] = (int32_t)((int64_t)a.B * a.g.E);
  }
}

__global__ void __launch_bounds__(256) build_grid_graph_kernel(const GridBuildArgs a) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < a.endD; it += stride) {
    if (it < a.endA) {
      if (a.patch) phase_patch_features(a, it); else phase_pixel_features(a, it);
    } else if (it < a.endB) {
      phase_positions(a, it - a.endA);
    } else if (it < a.endC) {
      phase_edges(a, it - a.endB);
    } else {
      phase_csr(a, it - a.endC);
    }
  }
}

// family of every edge of a batched grid graph: 0 horizontal, 1 vertical, 2 / 3 the diagonals.
// All edges of a family share one geometry row [d_row, d_col, L1] (SURVEY.md section 0.4).
__global__ void grid_edge_class_kernel(GridDims g, int64_t BE, int32_t* __restrict__ cls) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t ge = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; ge < BE; ge += stride) {
    const int64_t e = ge % g.E;
    cls[ge] = e < g.Eh ? 0 : (e < g.Eh + g.Ev ? 1 : (e < g.Eh + g.Ev + g.Ed ? 2 : 3));
  }
}

// paired destination slots of a batched grid graph without diagonals (grid_slot_src): for slot s of 2 B N, its source
// node (-1: padding slot), its destination node s >> 1 and its edge class (0 horizontal, 1 vertical: the slot's parity)
__global__ void grid_pair_slots_kernel(GridDims g, int64_t BS, int32_t* __restrict__ src, int32_t* __restrict__ dst,
                                       int32_t* __restrict__ cls) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < BS; s += stride) {
    const int64_t b = s / (2 * g.N), local = grid_slot_src(g, s - b * 2 * g.N);
    src[s] = local < 0 ? -1 : (int32_t)(b * g.N + local);
    dst[s] = (int32_t)(s >> 1);
    cls[s] = (int32_t)(s & 1);
  }
}

static int launch_grid_build(const uint8_t* img, int B, int imgH, int imgW, int patch, int diagonals,
                             float* x, float* pos, int64_t* ei, int32_t* src32, int32_t* dst32,
                             int32_t* drp, int32_t* deid, int32_t* srp, int32_t* seid, cudaStream_t st) {
  GNC_REQUIRE(B > 0 && imgH > 0 && imgW > 0, "build graph: B, H, W must be positive");
  GNC_REQUIRE(img && x, "build graph: img and x must be non-null");
  const bool any_csr = src32 || dst32 || drp || deid || srp || seid;
  const bool all_csr = src32 && dst32 && drp && deid && srp && seid;
  GNC_REQUIRE(!any_csr || all_csr, "build graph: pass all six CSR arrays or none");
  GridBuildArgs a;
  a.img = img; a.x = x; a.pos = pos; a.ei = ei;
  a.src32 = src32; a.dst32 = dst32; a.drp = drp; a.deid = deid; a.srp = srp; a.seid = seid;
  a.B = B; a.imgH = imgH; a.imgW = imgW; a.patch = patch;
  if (patch) {
    GNC_REQUIRE(patch > 0 && imgH / patch > 0 && imgW / patch > 0, "patch graph: patch larger than image");
    a.g = make_grid(imgH / patch, imgW / patch, 0);
  } else {
    a.g = make_grid(imgH, imgW, diagonals ? 1 : 0);
  }
  const int64_t BN = (int64_t)B * a.g.N, BE = (int64_t)B * a.g.E;
  GNC_REQUIRE(BN < 2147483647LL && BE < 2147483647LL, "build graph: B*N and B*E must fit int32");
  a.vecA = (!patch && aligned16(img) && aligned16(x)) ? 1 : 0;
  // pixel features: whole warps of 16-byte units (the lanes of a warp share a 512-byte block, phase_pixel_features)
  const int64_t nA = patch ? BN : (a.vecA ? ceil_div<int64_t>(ceil_div<int64_t>(BN * 3, 16), 32) * 32 : ceil_div<int64_t>(BN * 3, 16));
  a.endA = nA;
  a.endB = a.endA + (pos ? BN : 0);
  a.endC = a.endB + ((ei || all_csr) ? BE : 0);
  a.endD = a.endC + (all_csr ? BN : 0);
  const int64_t blocks_needed = ceil_div<int64_t>(a.endD, 256);
  int64_t blocks = blocks_needed < (int64_t)kNumSMs * 16 ? blocks_needed : (int64_t)kNumSMs * 16;
  if (blocks < 1) blocks = 1;
  build_grid_graph_kernel<<<(unsigned)blocks, 256, 0, st>>>(a);
  return check_launch("build_grid_graph_kernel");
}

// ----------------------------------------------------------------------------
// Generic stable CSR: histogram -> exclusive scan -> fill -> per-row sort.
// ----------------------------------------------------------------------------
__global__ void csr_histogram_kernel(const int64_t* __restrict__ key, int64_t kstride, int64_t E, int64_t N,
                                     int32_t* __restrict__ cnt, int32_t* __restrict__ key32,
                                     int32_t* __restrict__ bad) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += stride) {
    const int64_t k = key[e * kstride];
    if (k < 0 || k >= N) {
      if (bad) atomicExch(bad, 1);
      if (key32) key32[e] = 0;
      continue;
    }
    if (key32) key32[e] = (int32_t)k;
    atomicAdd(cnt + k, 1);
  }
}

constexpr int kScanThreads = 512;
constexpr int kScanItems = 4;
constexpr int kScanTile = kScanThreads * kScanItems;

// In-place exclusive scan of one tile per block; block totals to sums[].
__global__ void __launch_bounds__(kScanThreads) scan_tiles_kernel(int32_t* __restrict__ data, int64_t n,
                                                                  int32_t* __restrict__ sums) {
  __shared__ int32_t warp_tot[kScanThreads / 32];
  const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  int32_t v[kScanItems];
  int32_t t = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    v[i] = (base + i < n) ? data[base + i] : 0;
    t += v[i];
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int32_t inc = t;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int32_t u = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += u;
  }
  if (lane == 31) warp_tot[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int32_t w = (lane < kScanThreads / 32) ? warp_tot[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int32_t u = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += u;
    }
    if (lane < kScanThreads / 32) warp_tot[lane] = w;   // inclusive over warps
  }
  __syncthreads();
  int32_t excl = inc - t + (warp > 0 ? warp_tot[warp - 1] : 0);
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    if (base + i < n) data[base + i] = excl;
    excl += v[i];
  }
  if (threadIdx.x == kScanThreads - 1 && sums) sums[blockIdx.x] = warp_tot[kScanThreads / 32 - 1];
}

__global__ void __launch_bounds__(kScanThreads) scan_add_kernel(int32_t* __restrict__ data, int64_t n,
                                                                const int32_t* __restrict__ sums) {
  const int32_t add = sums[blockIdx.x];
  const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i)
    if (base + i < n) data[base + i] += add;
}

// exclusive scan of data[0..n) in place; scratch needs >= n/kScanTile + 2 levels.
static int exclusive_scan_i32(int32_t* data, int64_t n, int32_t* scratch, cudaStream_t st) {
  const int64_t tiles = ceil_div<int64_t>(n, kScanTile);
  if (tiles <= 1) {
    scan_tiles_kernel<<<1, kScanThreads, 0, st>>>(data, n, nullptr);
    return check_launch("scan_tiles_kernel");
  }
  scan_tiles_kernel<<<(unsigned)tiles, kScanThreads, 0, st>>>(data, n, scratch);
  int rc = check_launch("scan_tiles_kernel");
  if (rc) return rc;
  rc = exclusive_scan_i32(scratch, tiles, scratch + tiles, st);
  if (rc) return rc;
  scan_add_kernel<<<(unsigned)tiles, kScanThreads, 0, st>>>(data, n, scratch);
  return check_launch("scan_add_kernel");
}

__global__ void csr_fill_kernel(const int64_t* __restrict__ key, int64_t kstride, int64_t E, int64_t N,
                                const int32_t* __restrict__ rowptr, int32_t* __restrict__ cursor,
                                int32_t* __restrict__ eid) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += stride) {
    const int64_t k = key[e * kstride];
    if (k < 0 || k >= N) continue;
    const int32_t slot = atomicAdd(cursor + k, 1);
    eid[rowptr[k] + slot] = (int32_t)e;
  }
}

// Slots inside a row were claimed in arbitrary order; restore ascending edge id
// (the summation order of the CPU reference).  Rows are short on every graph this
// path builds (<= 4 on grids, ~6 on superpixels); long rows fall back to heapsort.
__global__ void csr_sort_rows_kernel(const int32_t* __restrict__ rowptr, int64_t N, int32_t* __restrict__ eid) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < N; v += stride) {
    const int32_t s = rowptr[v], n = rowptr[v + 1] - s;
    if (n < 2) continue;
    int32_t* a = eid + s;
    if (n <= 32) {
      for (int i = 1; i < n; ++i) {
        const int32_t x = a[i];
        int j = i - 1;
        while (j >= 0 && a[j] > x) { a[j + 1] = a[j]; --j; }
        a[j + 1] = x;
      }
    } else {
      for (int start = n / 2 - 1; start >= 0; --start) {      // heapify
        int root = start;
        for (;;) {
          int child = 2 * root + 1;
          if (child >= n) break;
          if (child + 1 < n && a[child] < a[child + 1]) ++child;
          if (a[root] >= a[child]) break;
          int32_t t = a[root]; a[root] = a[child]; a[child] = t;
          root = child;
        }
      }
      for (int end = n - 1; end > 0; --end) {
        int32_t t = a[0]; a[0] = a[end]; a[end] = t;
        int root = 0;
        for (;;) {
          int child = 2 * root + 1;
          if (child >= end) break;
          if (child + 1 < end && a[child] < a[child + 1]) ++child;
          if (a[root] >= a[child]) break;
          int32_t u = a[root]; a[root] = a[child]; a[child] = u;
          root = child;
        }
      }
    }
  }
}

// ----------------------------------------------------------------------------
// Label map -> superpixel graph.  One CTA per image; integer statistics are
// accumulated with shared-memory atomics (exact, order-independent).
// ----------------------------------------------------------------------------
__global__ void __launch_bounds__(256) superpixel_graph_kernel(
    const uint8_t* __restrict__ img, const int32_t* __restrict__ labels, int H, int W, int max_label,
    int S_max, int64_t E_max, int32_t* __restrict__ n_nodes, float* __restrict__ x, float* __restrict__ pos,
    uint8_t* __restrict__ adj, int32_t* __restrict__ n_edges, int64_t* __restrict__ edges,
    int32_t* __restrict__ work, int64_t work_per_image, int use_smem, int32_t* __restrict__ bad) {
  extern __shared__ int32_t sp_smem[];
  const int b = blockIdx.x;
  const int64_t HW = (int64_t)H * W;
  const uint8_t* im = img + (int64_t)b * HW * 3;
  const int32_t* lab = labels + (int64_t)b * HW;
  // scratch layout: rank[max_label+1] | cnt,s_r,s_g,s_b,s_row,s_col [6][S_max] (uint32; 64-bit hi parts
  // are not needed: 255 * 2^24 pixels < 2^32 and row/col sums < 2^12 * 2^24) | rowoff[S_max+1].
  // It lives in shared memory when it fits (the usual ~100 superpixels), else in the global workspace.
  int32_t* rank = use_smem ? sp_smem : work + (int64_t)b * work_per_image;
  uint32_t* stat = reinterpret_cast<uint32_t*>(rank + (max_label + 1));
  int32_t* rowoff = reinterpret_cast<int32_t*>(stat + 6 * (int64_t)S_max);
  uint8_t* A = adj + (int64_t)b * S_max * S_max;
  __shared__ int s_S;

  for (int l = threadIdx.x; l <= max_label; l += blockDim.x) rank[l] = 0;
  for (int i = threadIdx.x; i < 6 * S_max; i += blockDim.x) stat[i] = 0;
  __syncthreads();
  for (int64_t p = threadIdx.x; p < HW; p += blockDim.x) {
    const int32_t l = lab[p];
    if (l < 0 || l > max_label) { if (bad) atomicExch(bad, 1); continue; }
    rank[l] = 1;                                        // benign race: all writers store 1
  }
  __syncthreads();
  if (threadIdx.x == 0) {                               // rank among present labels (np.unique order)
    int r = 0;
    for (int l = 0; l <= max_label; ++l) {
      const int present = rank[l];
      rank[l] = present ? r : -1;
      r += present;
    }
    s_S = r;
    n_nodes[b] = r;
    if (r > S_max && bad) atomicExch(bad, 2);
  }
  __syncthreads();
  const int S = s_S < S_max ? s_S : S_max;
  for (int64_t p = threadIdx.x; p < HW; p += blockDim.x) {
    const int32_t l = lab[p];
    if (l < 0 || l > max_label) continue;
    const int s = rank[l];
    if (s >= S_max) continue;
    const int r = (int)(p / W), c = (int)(p - (int64_t)r * W);
    atomicAdd(stat + 0 * S_max + s, 1u);
    atomicAdd(stat + 1 * S_max + s, (uint32_t)im[p * 3 + 0]);
    atomicAdd(stat + 2 * S_max + s, (uint32_t)im[p * 3 + 1]);
    atomicAdd(stat + 3 * S_max + s, (uint32_t)im[p * 3 + 2]);
    atomicAdd(stat + 4 * S_max + s, (uint32_t)r);
    atomicAdd(stat + 5 * S_max + s, (uint32_t)c);
    // 4-connected adjacency == default binary_dilation cross (superpixel.py:62-64)
    if (c + 1 < W) {
      const int32_t l2 = lab[p + 1];
      if (l2 != l && l2 >= 0 && l2 <= max_label) {
        const int t = rank[l2];
        if (t < S_max) { A[(int64_t)s * S_max + t] = 1; A[(int64_t)t * S_max + s] = 1; }
      }
    }
    if (r + 1 < H) {
      const int32_t l2 = lab[p + W];
      if (l2 != l && l2 >= 0 && l2 <= max_label) {
        const int t = rank[l2];
        if (t < S_max) { A[(int64_t)s * S_max + t] = 1; A[(int64_t)t * S_max + s] = 1; }
      }
    }
  }
  __syncthreads();
  __threadfence_block();
  for (int s = threadIdx.x; s < S; s += blockDim.x) {
    const double n = (double)stat[s];
    float* xo = x + ((int64_t)b * S_max + s) * 3;
    // mean of img/255 over the segment; exact integer sums, float64 arithmetic,
    // then the loader's float32 cast (superpixel.py:43, dataloader.py:49)
    xo[0] = (float)(((double)stat[1 * S_max + s] / 255.0) / n);
    xo[1] = (float)(((double)stat[2 * S_max + s] / 255.0) / n);
    xo[2] = (float)(((double)stat[3 * S_max + s] / 255.0) / n);
    float* po = pos + ((int64_t)b * S_max + s) * 2;
    po[0] = (float)((double)stat[4 * S_max + s] / n);
    po[1] = (float)((double)stat[5 * S_max + s] / n);
    int cnt = 0;
    for (int t = s + 1; t < S; ++t) cnt += A[(int64_t)s * S_max + t];
    rowoff[s] = cnt;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int acc = 0;
    for (int s = 0; s < S; ++s) { const int c = rowoff[s]; rowoff[s] = acc; acc += c; }
    rowoff[S] = acc;
    n_edges[b] = 2 * acc;
    if (2 * (int64_t)acc > E_max && bad) atomicExch(bad, 3);
  }
  __syncthreads();
  int64_t* e0 = edges + (int64_t)b * 2 * E_max;
  int64_t* e1 = e0 + E_max;
  for (int s = threadIdx.x; s < S; s += blockDim.x) {
    int64_t k = 2 * (int64_t)rowoff[s];
    for (int t = s + 1; t < S; ++t) {
      if (A[(int64_t)s * S_max + t]) {
        if (k + 1 < E_max) {
          e0[k] = s; e1[k] = t;                         // (i, j)
          e0[k + 1] = t; e1[k + 1] = s;                 // (j, i)
        }
        k += 2;
      }
    }
  }
}


// The same stage for widths that are a multiple of 8 (every resize the reference uses): 1024 threads per image, a thread
// owns 8 consecutive pixels of a row (labels as two 128-bit loads, pixels as three 64-bit loads) and a warp an
// 8-pixel-wide strip of 32 rows, so its lanes meet only a few labels.  The integer statistics of a thread's label run
// are merged per label across the warp (match.any + redux.sync) before they go to the shared-memory atomics: a few
// atomics per warp and row strip instead of six contended atomics per pixel.  Same sums, same outputs as the kernel
// above (tests/test_gpu_graph_build.py runs both against the oracle).
__global__ void __launch_bounds__(1024) superpixel_graph_run8_kernel(
    const uint8_t* __restrict__ img, const int32_t* __restrict__ labels, int H, int W, int max_label,
    int S_max, int64_t E_max, int32_t* __restrict__ n_nodes, float* __restrict__ x, float* __restrict__ pos,
    uint8_t* __restrict__ adj, int32_t* __restrict__ n_edges, int64_t* __restrict__ edges,
    int32_t* __restrict__ work, int64_t work_per_image, int use_smem, int32_t* __restrict__ bad) {
  extern __shared__ int32_t sp_smem[];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
  const int64_t HW = (int64_t)H * W;
  const uint8_t* im = img + (int64_t)b * HW * 3;
  const int32_t* lab = labels + (int64_t)b * HW;
  int32_t* rank = use_smem ? sp_smem : work + (int64_t)b * work_per_image;
  uint32_t* stat = reinterpret_cast<uint32_t*>(rank + (max_label + 1));
  int32_t* rowoff = reinterpret_cast<int32_t*>(stat + 6 * (int64_t)S_max);
  uint8_t* A = adj + (int64_t)b * S_max * S_max;
  __shared__ int s_S;

  for (int l = tid; l <= max_label; l += blockDim.x) rank[l] = 0;
  for (int i = tid; i < 6 * S_max; i += blockDim.x) stat[i] = 0;
  __syncthreads();
  for (int64_t q = tid; q < HW / 4; q += blockDim.x) {                  // labels present (coalesced 128-bit reads)
    const int4 v = __ldg(reinterpret_cast<const int4*>(lab) + q);
    const int l4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (l4[j] < 0 || l4[j] > max_label) { if (bad) atomicExch(bad, 1); continue; }
      if (rank[l4[j]] == 0) rank[l4[j]] = 1;                            // benign race: all writers store 1
    }
  }
  __syncthreads();
  if (tid == 0) {                                                       // rank among present labels (np.unique order)
    int r = 0;
    for (int l = 0; l <= max_label; ++l) {
      const int present = rank[l];
      rank[l] = present ? r : -1;
      r += present;
    }
    s_S = r;
    n_nodes[b] = r;
    if (r > S_max && bad) atomicExch(bad, 2);
  }
  __syncthreads();
  const int S = s_S < S_max ? s_S : S_max;
  auto node_of = [&](int32_t l) { return (l < 0 || l > max_label) ? -1 : rank[l]; };
  auto link = [&](int s, int32_t l2) {                                  // 4-connected adjacency (superpixel.py:62-64)
    const int t = node_of(l2);
    if (t >= 0 && t != s && t < S_max) { A[(int64_t)s * S_max + t] = 1; A[(int64_t)t * S_max + s] = 1; }
  };
  auto add_stats = [&](int s, unsigned n, unsigned r, unsigned g, unsigned bl, unsigned row, unsigned col) {
    atomicAdd(stat + 0 * S_max + s, n); atomicAdd(stat + 1 * S_max + s, r); atomicAdd(stat + 2 * S_max + s, g);
    atomicAdd(stat + 3 * S_max + s, bl); atomicAdd(stat + 4 * S_max + s, row); atomicAdd(stat + 5 * S_max + s, col);
  };
  const int gpr = W >> 3;
  const int G = ((H + 31) >> 5) * 32 * gpr;
  for (int base = 0; base < G; base += blockDim.x) {                    // warp-uniform trip count
    const int gi = base + tid;
    const int band = gi / (gpr * 32), rem = gi - band * gpr * 32;
    const int y = band * 32 + (rem & 31), x0 = (rem >> 5) << 3;
    const bool active = y < H;
    int run_s = -1;
    unsigned cn = 0, cr = 0, cg = 0, cb = 0, ccol = 0;
    if (active) {
      const int64_t p0 = (int64_t)y * W + x0;
      const int4 la = __ldg(reinterpret_cast<const int4*>(lab + p0)), lb = __ldg(reinterpret_cast<const int4*>(lab + p0) + 1);
      const int32_t l8[8] = {la.x, la.y, la.z, la.w, lb.x, lb.y, lb.z, lb.w};
      uint32_t w[6];
      {
        const uint2* src = reinterpret_cast<const uint2*>(im + p0 * 3);
#pragma unroll
        for (int j = 0; j < 3; ++j) { const uint2 v = __ldg(src + j); w[2 * j] = v.x; w[2 * j + 1] = v.y; }
      }
      int32_t d8[8];
      const bool down = y + 1 < H;
      if (down) {
        const int4 da = __ldg(reinterpret_cast<const int4*>(lab + p0 + W)), db = __ldg(reinterpret_cast<const int4*>(lab + p0 + W) + 1);
        d8[0] = da.x; d8[1] = da.y; d8[2] = da.z; d8[3] = da.w; d8[4] = db.x; d8[5] = db.y; d8[6] = db.z; d8[7] = db.w;
      }
      const int32_t l_next = x0 + 8 < W ? __ldg(lab + p0 + 8) : l8[7];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int s = node_of(l8[i]);
        if (s < 0 || s >= S_max) continue;
        if (s != run_s) {
          if (cn) add_stats(run_s, cn, cr, cg, cb, cn * (unsigned)y, ccol);
          run_s = s; cn = cr = cg = cb = ccol = 0;
        }
        const int b0 = 3 * i, b1 = 3 * i + 1, b2 = 3 * i + 2;
        cn += 1;
        cr += (w[b0 >> 2] >> (8 * (b0 & 3))) & 255u;
        cg += (w[b1 >> 2] >> (8 * (b1 & 3))) & 255u;
        cb += (w[b2 >> 2] >> (8 * (b2 & 3))) & 255u;
        ccol += (unsigned)(x0 + i);
        const int32_t right = i < 7 ? l8[i + 1] : l_next;
        if (right != l8[i]) link(s, right);
        if (down && d8[i] != l8[i]) link(s, d8[i]);
      }
    }
    // the open runs of the warp's lanes, merged per node
    const unsigned peers = __match_any_sync(0xffffffffu, cn ? run_s : -1);
    const unsigned tn = __reduce_add_sync(peers, cn), tr = __reduce_add_sync(peers, cr), tg = __reduce_add_sync(peers, cg);
    const unsigned tb = __reduce_add_sync(peers, cb), trow = __reduce_add_sync(peers, cn * (unsigned)y);
    const unsigned tcol = __reduce_add_sync(peers, ccol);
    if (cn && lane == __ffs(peers) - 1) add_stats(run_s, tn, tr, tg, tb, trow, tcol);
  }
  __syncthreads();
  __threadfence_block();
  for (int s = tid; s < S; s += blockDim.x) {
    const double n = (double)stat[s];
    float* xo = x + ((int64_t)b * S_max + s) * 3;
    xo[0] = (float)(((double)stat[1 * S_max + s] / 255.0) / n);
    xo[1] = (float)(((double)stat[2 * S_max + s] / 255.0) / n);
    xo[2] = (float)(((double)stat[3 * S_max + s] / 255.0) / n);
    float* po = pos + ((int64_t)b * S_max + s) * 2;
    po[0] = (float)((double)stat[4 * S_max + s] / n);
    po[1] = (float)((double)stat[5 * S_max + s] / n);
    int cnt = 0;
    for (int t = s + 1; t < S; ++t) cnt += A[(int64_t)s * S_max + t];
    rowoff[s] = cnt;
  }
  __syncthreads();
  if (tid == 0) {
    int acc = 0;
    for (int s = 0; s < S; ++s) { const int c = rowoff[s]; rowoff[s] = acc; acc += c; }
    rowoff[S] = acc;
    n_edges[b] = 2 * acc;
    if (2 * (int64_t)acc > E_max && bad) atomicExch(bad, 3);
  }
  __syncthreads();
  int64_t* e0 = edges + (int64_t)b * 2 * E_max;
  int64_t* e1 = e0 + E_max;
  for (int s = tid; s < S; s += blockDim.x) {
    int64_t k = 2 * (int64_t)rowoff[s];
    for (int t = s + 1; t < S; ++t) {
      if (A[(int64_t)s * S_max + t]) {
        if (k + 1 < E_max) {
          e0[k] = s; e1[k] = t;
          e0[k + 1] = t; e1[k + 1] = s;
        }
        k += 2;
      }
    }
  }
}


// Block-diagonal batch of per-image superpixel graphs (different node / edge counts): offsets by one single-CTA scan,
// then one CTA per image copies its valid rows to their place and shifts the edge endpoints by the image's node offset.
__global__ void __launch_bounds__(1024) superpixel_offsets_kernel(const int32_t* __restrict__ n_nodes, const int32_t* __restrict__ n_edges,
                                                                  int B, int S_max, int64_t E_max, int32_t* __restrict__ node_ptr,
                                                                  int64_t* __restrict__ edge_ptr) {
  __shared__ long long s_n[1024], s_e[1024];
  const int t = threadIdx.x;
  const int per = (B + 1023) / 1024;
  long long an = 0, ae = 0;
  for (int i = t * per; i < min(B, (t + 1) * per); ++i) {
    an += min(n_nodes[i], S_max);
    ae += min((long long)n_edges[i], (long long)E_max);
  }
  s_n[t] = an; s_e[t] = ae;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {
    const long long vn = t >= off ? s_n[t - off] : 0, ve = t >= off ? s_e[t - off] : 0;
    __syncthreads();
    s_n[t] += vn; s_e[t] += ve;
    __syncthreads();
  }
  long long rn = s_n[t] - an, re = s_e[t] - ae;
  for (int i = t * per; i < min(B, (t + 1) * per); ++i) {
    node_ptr[i] = (int32_t)rn; edge_ptr[i] = re;
    rn += min(n_nodes[i], S_max);
    re += min((long long)n_edges[i], (long long)E_max);
  }
  if (t == 1023) { node_ptr[B] = (int32_t)s_n[1023]; edge_ptr[B] = s_e[1023]; }
}

__global__ void __launch_bounds__(256) superpixel_compact_kernel(const float* __restrict__ x, const float* __restrict__ pos,
                                                                 const int64_t* __restrict__ edges, int S_max, int64_t E_max,
                                                                 const int32_t* __restrict__ node_ptr, const int64_t* __restrict__ edge_ptr,
                                                                 float* __restrict__ xb, float* __restrict__ pb,
                                                                 int64_t* __restrict__ eb, int64_t e_total) {
  const int b = blockIdx.x;
  const int n0 = node_ptr[b], nn = node_ptr[b + 1] - n0;
  const int64_t e0 = edge_ptr[b], ne = edge_ptr[b + 1] - e0;
  const float* xs = x + (int64_t)b * S_max * 3;
  const float* ps = pos + (int64_t)b * S_max * 2;
  for (int i = threadIdx.x; i < nn * 3; i += blockDim.x) xb[(int64_t)n0 * 3 + i] = xs[i];
  for (int i = threadIdx.x; i < nn * 2; i += blockDim.x) pb[(int64_t)n0 * 2 + i] = ps[i];
  const int64_t* es = edges + (int64_t)b * 2 * E_max;
  for (int64_t i = threadIdx.x; i < ne; i += blockDim.x) {
    eb[e0 + i] = es[i] + n0;
    eb[e_total + e0 + i] = es[E_max + i] + n0;
  }
}

// The same batch at host-known sizes (N_alloc = B * S_cap + 1 rows, E_alloc = B * E_cap edges), so that nothing has to
// be read back and the build can be captured in a CUDA graph.  Rows [0, node_ptr[B]) and edges [0, edge_ptr[B]) are what
// superpixel_compact_kernel writes.  The padding rows [P0, N_alloc) are zero and padding edge P0 + k is a self-loop of
// padding row P0 + k mod (N_alloc - P0): no real row meets a padding edge, and the padding rows' in-degrees stay near
// E_pad / N_pad, which keeps the CSR build's per-row sort and the aggregation's per-row loop short.  Every offset is
// clamped to the buffers, so nothing is written out of bounds whatever the inputs hold; what does not fit is reported
// in *overflow (bit 0: a label outside [0, max_label], bit 1: more than S_cap nodes, bit 2: more than E_cap edges).
__global__ void __launch_bounds__(256) superpixel_padded_kernel(
    const float* __restrict__ x, const float* __restrict__ pos, const int64_t* __restrict__ edges,
    const int32_t* __restrict__ n_nodes, const int32_t* __restrict__ n_edges, const int32_t* __restrict__ labels,
    int B, int64_t HW, int max_label, int S_cap, int64_t E_cap, const int32_t* __restrict__ node_ptr,
    const int64_t* __restrict__ edge_ptr, float* __restrict__ xb, float* __restrict__ pb, int64_t* __restrict__ eb,
    int32_t* __restrict__ overflow) {
  const int64_t N_alloc = (int64_t)B * S_cap + 1, E_alloc = (int64_t)B * E_cap;
  auto clamp = [](int64_t v, int64_t lo, int64_t hi) { return v < lo ? lo : (v > hi ? hi : v); };
  int bad = 0;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    if (n_nodes[b] > S_cap) bad |= 2;
    if (n_edges[b] > E_cap) bad |= 4;
    const int64_t n0 = clamp(node_ptr[b], 0, N_alloc - 1);
    const int64_t nn = clamp((int64_t)node_ptr[b + 1] - node_ptr[b], 0, S_cap < N_alloc - 1 - n0 ? S_cap : N_alloc - 1 - n0);
    const int64_t e0 = clamp(edge_ptr[b], 0, E_alloc);
    const int64_t ne = clamp(edge_ptr[b + 1] - edge_ptr[b], 0, E_cap < E_alloc - e0 ? E_cap : E_alloc - e0);
    const float* xs = x + (int64_t)b * S_cap * 3;
    const float* ps = pos + (int64_t)b * S_cap * 2;
    for (int64_t i = threadIdx.x; i < nn * 3; i += blockDim.x) xb[n0 * 3 + i] = xs[i];
    for (int64_t i = threadIdx.x; i < nn * 2; i += blockDim.x) pb[n0 * 2 + i] = ps[i];
    const int64_t* es = edges + (int64_t)b * 2 * E_cap;
    for (int64_t i = threadIdx.x; i < ne; i += blockDim.x) {
      eb[e0 + i] = es[i] + n0;
      eb[E_alloc + e0 + i] = es[E_cap + i] + n0;
    }
  }
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nthreads = (int64_t)gridDim.x * blockDim.x;
  const int64_t P0 = clamp(node_ptr[B], 0, N_alloc - 1), Q0 = clamp(edge_ptr[B], 0, E_alloc);
  for (int64_t i = P0 * 3 + tid; i < N_alloc * 3; i += nthreads) xb[i] = 0.f;
  for (int64_t i = P0 * 2 + tid; i < N_alloc * 2; i += nthreads) pb[i] = 0.f;
  for (int64_t k = Q0 + tid; k < E_alloc; k += nthreads) {
    const int64_t v = P0 + (k - Q0) % (N_alloc - P0);
    eb[k] = v;
    eb[E_alloc + k] = v;
  }
  if (labels) {
    for (int64_t p = tid; p < (int64_t)B * HW; p += nthreads) {
      const int32_t l = labels[p];
      if (l < 0 || l > max_label) bad |= 1;
    }
  }
  if (bad) atomicOr(overflow, bad);
}

}  // namespace gnc

using namespace gnc;

extern "C" {

int gnc_version(void) { return 100; }
const char* gnc_last_error(void) { return g_err; }
uint64_t gnc_launch_count(void) { return g_launches.load(); }
void gnc_reset_launch_count(void) { g_launches.store(0); }

int64_t gnc_grid_num_edges(int H, int W, int diagonals) {
  if (H <= 0 || W <= 0) return 0;
  return make_grid(H, W, diagonals ? 1 : 0).E;
}

int gnc_build_pixel_graph_u8(const uint8_t* img, int B, int H, int W, int diagonals, float* x, float* pos,
                             int64_t* edge_index, int32_t* src32, int32_t* dst32, int32_t* dst_rowptr,
                             int32_t* dst_eid, int32_t* src_rowptr, int32_t* src_eid, gnc_stream_t stream) {
  return launch_grid_build(img, B, H, W, 0, diagonals, x, pos, edge_index, src32, dst32, dst_rowptr, dst_eid,
                           src_rowptr, src_eid, (cudaStream_t)stream);
}

int gnc_build_patch_graph_u8(const uint8_t* img, int B, int H, int W, int patch, float* x, float* pos,
                             int64_t* edge_index, int32_t* src32, int32_t* dst32, int32_t* dst_rowptr,
                             int32_t* dst_eid, int32_t* src_rowptr, int32_t* src_eid, gnc_stream_t stream) {
  GNC_REQUIRE(patch > 0, "patch graph: patch must be positive");
  return launch_grid_build(img, B, H, W, patch, 0, x, pos, edge_index, src32, dst32, dst_rowptr, dst_eid,
                           src_rowptr, src_eid, (cudaStream_t)stream);
}

int gnc_grid_edge_class(int B, int H, int W, int diagonals, int32_t* cls, gnc_stream_t stream) {
  GNC_REQUIRE(B > 0 && H > 0 && W > 0 && cls, "grid_edge_class: bad arguments");
  const GridDims g = make_grid(H, W, diagonals ? 1 : 0);
  const int64_t BE = (int64_t)B * g.E;
  if (BE == 0) return GNC_OK;
  int64_t blocks = ceil_div<int64_t>(BE, 256);
  if (blocks > (int64_t)kNumSMs * 16) blocks = (int64_t)kNumSMs * 16;
  grid_edge_class_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(g, BE, cls);
  return check_launch("grid_edge_class_kernel");
}

int gnc_grid_pair_slots(int B, int H, int W, int32_t* slot_src, int32_t* slot_dst, int32_t* slot_class, gnc_stream_t stream) {
  GNC_REQUIRE(B > 0 && H > 0 && W > 0 && slot_src && slot_dst && slot_class, "grid_pair_slots: bad arguments");
  const GridDims g = make_grid(H, W, 0);
  const int64_t BS = 2 * (int64_t)B * g.N;
  GNC_REQUIRE(BS <= INT32_MAX, "grid_pair_slots: more than 2^31 slots");
  int64_t blocks = ceil_div<int64_t>(BS, 256);
  if (blocks > (int64_t)kNumSMs * 16) blocks = (int64_t)kNumSMs * 16;
  grid_pair_slots_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(g, BS, slot_src, slot_dst, slot_class);
  return check_launch("grid_pair_slots_kernel");
}

int64_t gnc_superpixel_workspace(int S_max, int max_label) {
  return (int64_t)(max_label + 1) + 6 * (int64_t)S_max + (S_max + 1) + 8;
}

int gnc_build_superpixel_graph(const uint8_t* img, const int32_t* labels, int B, int H, int W, int max_label,
                               int S_max, int64_t E_max, int32_t* n_nodes, float* x, float* pos, uint8_t* adj,
                               int32_t* n_edges, int64_t* edges, int32_t* work, gnc_stream_t stream) {
  GNC_REQUIRE(B > 0 && H > 0 && W > 0 && S_max > 0 && max_label >= 0 && E_max >= 0, "superpixel: bad sizes");
  GNC_REQUIRE((int64_t)H * W <= (1 << 24), "superpixel: image larger than 2^24 pixels");
  GNC_REQUIRE(img && labels && n_nodes && x && pos && adj && n_edges && edges && work, "superpixel: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t wpi = gnc_superpixel_workspace(S_max, max_label);
  cudaError_t e = cudaMemsetAsync(adj, 0, (size_t)B * S_max * S_max, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(x, 0, (size_t)B * S_max * 3 * sizeof(float), st);
  if (e == cudaSuccess) e = cudaMemsetAsync(pos, 0, (size_t)B * S_max * 2 * sizeof(float), st);
  if (e == cudaSuccess) e = cudaMemsetAsync(edges, 0, (size_t)B * 2 * E_max * sizeof(int64_t), st);
  if (e != cudaSuccess) return fail(GNC_ECUDA, "superpixel memset: %s", cudaGetErrorString(e));
  const size_t smem = (size_t)wpi * sizeof(int32_t);
  const int use_smem = smem <= 40 * 1024 ? 1 : 0;
  static const bool force_scalar = getenv("GNC_SUPERPIXEL_SCALAR") != nullptr;      // debug: the per-pixel kernel
  if (W % 8 == 0 && !force_scalar && ((reinterpret_cast<uintptr_t>(img) | reinterpret_cast<uintptr_t>(labels)) & 15u) == 0) {
    superpixel_graph_run8_kernel<<<B, 1024, use_smem ? smem : 0, st>>>(img, labels, H, W, max_label, S_max, E_max, n_nodes,
                                                                       x, pos, adj, n_edges, edges, work, wpi, use_smem, nullptr);
    return check_launch("superpixel_graph_run8_kernel");
  }
  superpixel_graph_kernel<<<B, 256, use_smem ? smem : 0, st>>>(img, labels, H, W, max_label, S_max, E_max, n_nodes, x,
                                                               pos, adj, n_edges, edges, work, wpi, use_smem, nullptr);
  return check_launch("superpixel_graph_kernel");
}

int gnc_superpixel_batch_offsets(const int32_t* n_nodes, const int32_t* n_edges, int B, int S_max, int64_t E_max,
                                 int32_t* node_ptr, int64_t* edge_ptr, gnc_stream_t stream) {
  GNC_REQUIRE(n_nodes && n_edges && node_ptr && edge_ptr && B > 0 && S_max > 0 && E_max >= 0, "superpixel_batch_offsets: bad arguments");
  superpixel_offsets_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(n_nodes, n_edges, B, S_max, E_max, node_ptr, edge_ptr);
  return check_launch("superpixel_offsets_kernel");
}

int gnc_superpixel_batch_compact(const float* x, const float* pos, const int64_t* edges, int B, int S_max, int64_t E_max,
                                 const int32_t* node_ptr, const int64_t* edge_ptr, float* xb, float* pb, int64_t* eb,
                                 int64_t e_total, gnc_stream_t stream) {
  GNC_REQUIRE(x && pos && edges && node_ptr && edge_ptr && xb && pb && (eb || e_total == 0) && B > 0 && S_max > 0 && E_max >= 0 &&
              e_total >= 0, "superpixel_batch_compact: bad arguments");
  superpixel_compact_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(x, pos, edges, S_max, E_max, node_ptr, edge_ptr, xb, pb, eb, e_total);
  return check_launch("superpixel_compact_kernel");
}

int gnc_superpixel_batch_padded(const float* x, const float* pos, const int64_t* edges, const int32_t* n_nodes,
                                const int32_t* n_edges, const int32_t* labels, int B, int H, int W, int max_label,
                                int S_cap, int64_t E_cap, const int32_t* node_ptr, const int64_t* edge_ptr, float* xb,
                                float* pb, int64_t* eb, int32_t* overflow, gnc_stream_t stream) {
  GNC_REQUIRE(x && pos && edges && n_nodes && n_edges && node_ptr && edge_ptr && xb && pb && overflow && B > 0 && S_cap > 0 &&
              E_cap >= 0 && (eb || E_cap == 0) && (!labels || (H > 0 && W > 0 && max_label >= 0)),
              "superpixel_batch_padded: bad arguments");
  GNC_REQUIRE((int64_t)B * S_cap + 1 < INT32_MAX && (int64_t)B * E_cap < INT32_MAX,
              "superpixel_batch_padded: node and edge counts must fit int32");
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(overflow, 0, sizeof(int32_t), st);
  if (e != cudaSuccess) return fail(GNC_ECUDA, "superpixel_batch_padded memset: %s", cudaGetErrorString(e));
  const int64_t HW = labels ? (int64_t)H * W : 0;
  const int64_t work = (int64_t)B * (HW + E_cap + 3 * S_cap);
  const int64_t blocks = std::max<int64_t>(B, std::min<int64_t>(ceil_div<int64_t>(work, 256 * 8), (int64_t)kNumSMs * 4));
  superpixel_padded_kernel<<<(unsigned)blocks, 256, 0, st>>>(x, pos, edges, n_nodes, n_edges, labels, B, HW, max_label, S_cap,
                                                              E_cap, node_ptr, edge_ptr, xb, pb, eb, overflow);
  return check_launch("superpixel_padded_kernel");
}

int64_t gnc_csr_workspace(int64_t N) { return N + (N + 1) / 1024 + 64; }

int gnc_csr_build(const int64_t* key, int64_t key_stride, int64_t E, int64_t N, int32_t* rowptr, int32_t* eid,
                  int32_t* key32, int32_t* work, int32_t* bad, gnc_stream_t stream) {
  GNC_REQUIRE(E >= 0 && N >= 0 && N < 2147483647LL && E < 2147483647LL, "csr_build: E, N must fit int32");
  GNC_REQUIRE(rowptr && work && (E == 0 || (key && eid)), "csr_build: null pointer");
  GNC_REQUIRE(key_stride >= 1, "csr_build: key stride must be >= 1");
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(rowptr, 0, (size_t)(N + 1) * sizeof(int32_t), st);
  if (e == cudaSuccess && N > 0) e = cudaMemsetAsync(work, 0, (size_t)N * sizeof(int32_t), st);
  if (e != cudaSuccess) return fail(GNC_ECUDA, "csr_build memset: %s", cudaGetErrorString(e));
  int rc = GNC_OK;
  if (E > 0) {
    int64_t blocks = ceil_div<int64_t>(E, 256);
    if (blocks > (int64_t)kNumSMs * 16) blocks = (int64_t)kNumSMs * 16;
    csr_histogram_kernel<<<(unsigned)blocks, 256, 0, st>>>(key, key_stride, E, N, rowptr, key32, bad);
    if ((rc = check_launch("csr_histogram_kernel"))) return rc;
  }
  if ((rc = exclusive_scan_i32(rowptr, N + 1, work + N, st))) return rc;
  if (E > 0) {
    int64_t blocks = ceil_div<int64_t>(E, 256);
    if (blocks > (int64_t)kNumSMs * 16) blocks = (int64_t)kNumSMs * 16;
    csr_fill_kernel<<<(unsigned)blocks, 256, 0, st>>>(key, key_stride, E, N, rowptr, work, eid);
    if ((rc = check_launch("csr_fill_kernel"))) return rc;
    int64_t rblocks = ceil_div<int64_t>(N, 256);
    if (rblocks > (int64_t)kNumSMs * 16) rblocks = (int64_t)kNumSMs * 16;
    csr_sort_rows_kernel<<<(unsigned)rblocks, 256, 0, st>>>(rowptr, N, eid);
    if ((rc = check_launch("csr_sort_rows_kernel"))) return rc;
  }
  return GNC_OK;
}

}  // extern "C"
