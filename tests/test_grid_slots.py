"""CPU: the paired destination slots of csrc/grid_topology.h against the edge list of the numpy oracle.  Slot 2v holds
the in-edge of node v with the smaller edge id (horizontal), slot 2v+1 the other (vertical); -1 marks a missing edge."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import graph_build as ogb

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def harness():
    out = os.path.join(tempfile.gettempdir(), f"gnc_slots_harness_{os.getuid()}.so")
    src = os.path.join(HERE, "cpu_harness", "grid_slots_harness.cpp")
    subprocess.check_call(["g++", "-O1", "-shared", "-fPIC", "-o", out, src])
    return ctypes.CDLL(out)


@pytest.mark.parametrize("H,W", [(1, 1), (1, 5), (5, 1), (2, 2), (3, 7), (8, 5), (16, 16), (33, 17)])
def test_slots_match_edge_list(harness, H, W):
    ei = ogb.grid_edges(H, W, False)
    N = H * W
    edge, src = np.zeros(2 * N, np.int64), np.zeros(2 * N, np.int64)
    harness.harness_slots(H, W, edge.ctypes.data_as(ctypes.c_void_p), src.ctypes.data_as(ctypes.c_void_p))
    # every edge sits in exactly one slot, next to the other in-edge of its destination
    real = edge >= 0
    assert np.array_equal(np.sort(edge[real]), np.arange(ei.shape[1]))
    assert np.array_equal(src < 0, ~real)
    slots = np.nonzero(real)[0]
    assert np.array_equal(ei[1, edge[real]], slots >> 1)
    assert np.array_equal(ei[0, edge[real]], src[real])
    # slot order within a node is ascending edge id (scatter_sum's summation order)
    both = real[0::2] & real[1::2]
    assert np.all(edge[0::2][both] < edge[1::2][both])
    # in-degree of every node equals its number of real slots
    indeg = np.bincount(ei[1], minlength=N) if ei.shape[1] else np.zeros(N, np.int64)
    assert np.array_equal(indeg, real[0::2].astype(int) + real[1::2].astype(int))
