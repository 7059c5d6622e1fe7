// CPU harness: exposes the paired-slot arithmetic of graphnet_classifier_b200/csrc/grid_topology.h to Python
// (ctypes) so that it can be checked against the edge list without a GPU.  Test code only.
#include "../../graphnet_classifier_b200/csrc/grid_topology.h"

extern "C" {

// grids without diagonals: edge id and source node of every slot s < 2N (-1: padding slot)
void harness_slots(int H, int W, long long* edge, long long* src) {
  gnc::GridDims g = gnc::make_grid(H, W, 0);
  for (int64_t s = 0; s < 2 * g.N; ++s) {
    edge[s] = gnc::grid_slot_edge(g, s);
    src[s] = gnc::grid_slot_src(g, s);
  }
}
}
