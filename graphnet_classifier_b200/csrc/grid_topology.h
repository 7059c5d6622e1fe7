// Closed-form topology of the reference's directed pixel grid.
//
// Restates create_grid_edges_optimized (reference
// utils/image_to_graph/image_to_graph_optimized.py:7-39) as index arithmetic so
// that edge lists AND their CSR (by destination / by source) can be emitted
// directly, with no sort.  Edge families in emission order:
//   h : (i,j)   -> (i,j+1)    ids [0, Eh)            id = i*(W-1) + j
//   v : (i,j)   -> (i+1,j)    ids [Eh, Eh+Ev)        id = Eh + i*W + j
//   d1: (i,j)   -> (i+1,j+1)  ids [Eh+Ev, +Ed)       id = .. + i*(W-1) + j
//   d2: (i,j+1) -> (i+1,j)    ids [Eh+Ev+Ed, +Ed)    id = .. + i*(W-1) + j
// Node id of pixel (i,j) is i*W + j.  Header is host+device so the arithmetic is
// unit-tested on the CPU against the numpy oracle (tests/test_grid_topology.py).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define GNC_HD __host__ __device__ __forceinline__
#else
#define GNC_HD inline
#endif

namespace gnc {

struct GridDims {
  int H, W, diag;
  int64_t N, Eh, Ev, Ed, E;
};

GNC_HD GridDims make_grid(int H, int W, int diag) {
  GridDims g;
  g.H = H; g.W = W; g.diag = diag;
  g.N = (int64_t)H * W;
  g.Eh = (int64_t)H * (W - 1);
  g.Ev = (int64_t)(H - 1) * W;
  g.Ed = diag ? (int64_t)(H - 1) * (W - 1) : 0;
  g.E = g.Eh + g.Ev + 2 * g.Ed;
  return g;
}

// endpoints of local edge e (0 <= e < E)
GNC_HD void grid_edge(const GridDims& g, int64_t e, int64_t& src, int64_t& dst) {
  const int W = g.W;
  if (e < g.Eh) {
    int64_t i = e / (W - 1), j = e - i * (W - 1);
    src = i * W + j; dst = src + 1;
  } else if (e < g.Eh + g.Ev) {
    src = e - g.Eh; dst = src + W;
  } else if (e < g.Eh + g.Ev + g.Ed) {
    int64_t k = e - g.Eh - g.Ev;
    int64_t i = k / (W - 1), j = k - i * (W - 1);
    src = i * W + j; dst = src + W + 1;
  } else {
    int64_t k = e - g.Eh - g.Ev - g.Ed;
    int64_t i = k / (W - 1), j = k - i * (W - 1);
    src = i * W + j + 1; dst = src + W - 1;
  }
}

// In-edges of node v=(i,j), ascending edge id.  Returns the count (<= 4), fills
// ids[], and *before = number of in-edges of all nodes < v (the CSR row start).
GNC_HD int grid_in_edges(const GridDims& g, int64_t v, int64_t ids[4], int64_t* before) {
  const int W = g.W;
  const int64_t i = v / W, j = v - i * W;
  int n = 0;
  if (j > 0) ids[n++] = i * (W - 1) + (j - 1);
  if (i > 0) ids[n++] = g.Eh + (v - W);
  if (g.diag && i > 0) {
    if (j > 0) ids[n++] = g.Eh + g.Ev + (i - 1) * (W - 1) + (j - 1);
    if (j < W - 1) ids[n++] = g.Eh + g.Ev + g.Ed + (i - 1) * (W - 1) + j;
  }
  int64_t jm1 = j > 0 ? j - 1 : 0;
  int64_t b = i * (W - 1) + jm1;                    // h edges into earlier nodes
  if (i > 0) {
    b += (i - 1) * (int64_t)W + j;                  // v
    if (g.diag) {
      b += (i - 1) * (int64_t)(W - 1) + jm1;        // d1 (targets have j' > 0)
      b += (i - 1) * (int64_t)(W - 1) + (j < W - 1 ? j : W - 1);  // d2 (targets have j' < W-1)
    }
  }
  *before = b;
  return n;
}

// Out-edges of node v=(i,j), ascending edge id; *before = out-edges of nodes < v.
GNC_HD int grid_out_edges(const GridDims& g, int64_t v, int64_t ids[4], int64_t* before) {
  const int W = g.W, H = g.H;
  const int64_t i = v / W, j = v - i * W;
  int n = 0;
  if (j < W - 1) ids[n++] = i * (W - 1) + j;
  if (i < H - 1) ids[n++] = g.Eh + v;
  if (g.diag && i < H - 1) {
    if (j < W - 1) ids[n++] = g.Eh + g.Ev + i * (W - 1) + j;
    if (j > 0) ids[n++] = g.Eh + g.Ev + g.Ed + i * (W - 1) + (j - 1);
  }
  int64_t jm1 = j > 0 ? j - 1 : 0;
  int64_t jc = j < W - 1 ? j : W - 1;
  int64_t b = i * (W - 1) + jc;                     // h sources have j' < W-1
  b += (i < H - 1) ? v : (int64_t)(H - 1) * W;      // v sources have i' < H-1
  if (g.diag) {
    int64_t full = (i < H - 1 ? i : H - 1) * (int64_t)(W - 1);
    b += full + (i < H - 1 ? jc : 0);               // d1 sources: i'<H-1, j'<W-1
    b += full + (i < H - 1 ? jm1 : 0);              // d2 sources: i'<H-1, j'>0
  }
  *before = b;
  return n;
}

// Paired destination slots (grids without diagonals, where a node has at most two in-edges).  Slot 2v holds the
// horizontal in-edge of node v (from v-1, edge id i*(W-1)+j-1), slot 2v+1 the vertical one (from v-W, edge id
// Eh+v-W): the slot order of the edge ids into v is their ascending order, so (0 + y[2v]) + y[2v+1] is
// scatter_sum's bit pattern.  A slot whose edge does not exist (j = 0, resp. i = 0) is a padding slot.
// Returns the local edge id held by slot s (0 <= s < 2N), or -1 for a padding slot.
GNC_HD int64_t grid_slot_edge(const GridDims& g, int64_t s) {
  const int W = g.W;
  const int64_t v = s >> 1, i = v / W, j = v - i * W;
  if ((s & 1) == 0) return j > 0 ? i * (W - 1) + (j - 1) : -1;
  return i > 0 ? g.Eh + (v - W) : -1;
}

// Source node of slot s, or -1 for a padding slot.  The destination node of slot s is s >> 1.
GNC_HD int64_t grid_slot_src(const GridDims& g, int64_t s) {
  const int64_t v = s >> 1, i = v / g.W, j = v - i * g.W;
  if ((s & 1) == 0) return j > 0 ? v - 1 : -1;
  return i > 0 ? v - g.W : -1;
}

}  // namespace gnc
