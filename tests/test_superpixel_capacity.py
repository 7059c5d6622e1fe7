"""CPU: the per-image node / edge capacities of the captured superpixel path (batched.superpixel_capacity) against the
connectivity post-pass's rule restated on the CPU, and the planar edge bound against graphs that reach it."""
import itertools

import numpy as np
import pytest

from graphnet_classifier_b200.utils.image_to_graph.batched import superpixel_capacity


def _components(lab):
    """4-connected components of equal labels, numbered in scan order of their first pixel; and their sizes."""
    H, W = lab.shape
    comp = -np.ones((H, W), dtype=np.int64)
    sizes = []
    for y, x in itertools.product(range(H), range(W)):
        if comp[y, x] >= 0:
            continue
        c = len(sizes)
        stack, comp[y, x], n = [(y, x)], c, 0
        while stack:
            a, b = stack.pop()
            n += 1
            for u, v in ((a - 1, b), (a + 1, b), (a, b - 1), (a, b + 1)):
                if 0 <= u < H and 0 <= v < W and comp[u, v] < 0 and lab[u, v] == lab[a, b]:
                    comp[u, v] = c
                    stack.append((u, v))
        sizes.append(n)
    return comp, sizes


def _post_pass(lab, min_size):
    """csrc/slic_connect.cu steps 1-4: components smaller than min_size dissolve into the component left of (above, in
    column 0) their first pixel; the component of pixel 0 is always kept."""
    comp, sizes = _components(lab)
    H, W = lab.shape
    first = {}
    for y, x in itertools.product(range(H), range(W)):
        first.setdefault(comp[y, x], (y, x))
    tgt = list(range(len(sizes)))
    for c, (y, x) in first.items():
        if sizes[c] < min_size:
            if x > 0:
                tgt[c] = comp[y, x - 1]
            elif y > 0:
                tgt[c] = comp[y - 1, x]

    def root(c):
        while tgt[c] != c:
            c = tgt[c]
        return c
    kept = sorted({root(c) for c in range(len(sizes))})
    ids = {c: i for i, c in enumerate(kept)}
    return np.vectorize(lambda c: ids[root(c)])(comp)


def _adjacent_pairs(lab):
    pairs = set()
    for a, b in ((lab[:, :-1], lab[:, 1:]), (lab[:-1, :], lab[1:, :])):
        m = a != b
        pairs |= {(min(u, v), max(u, v)) for u, v in zip(a[m].tolist(), b[m].tolist())}
    return pairs


def test_capacity_formula():
    assert superpixel_capacity(256, 256, 327) == (201, 6 * 201 - 12)
    assert superpixel_capacity(8, 8, 0) == (64, 6 * 64 - 12)           # min_size 0: every component survives
    assert superpixel_capacity(4, 4, 1) == (16, 6 * 16 - 12)
    assert superpixel_capacity(1, 1, 0) == (1, 0)
    assert superpixel_capacity(1, 2, 0) == (2, 2)
    assert superpixel_capacity(3, 1, 5) == (1, 0)                     # min_size larger than the image: one region
    for S in range(1, 8):                                              # E_cap never exceeds the complete graph's edges
        E = superpixel_capacity(1, S, 0)[1]
        assert E <= S * (S - 1) and (S > 4 or E == S * (S - 1))        # K1 .. K4 are planar: the bound is reached


@pytest.mark.parametrize("H,W,min_size,k", [(12, 12, 0, 40), (12, 12, 3, 40), (9, 14, 5, 25), (16, 16, 8, 12),
                                            (7, 23, 2, 60), (20, 20, 20, 6)])
def test_post_pass_outputs_stay_within_capacity(H, W, min_size, k):
    """Label maps with many small, disconnected k-means-like segments (Voronoi cells of random seeds plus noise):
    after the post-pass every image has at most S_cap regions, each region is one 4-connected component, and the
    region adjacency graph has at most E_cap directed edges."""
    rng = np.random.default_rng(H * 1000 + W * 10 + min_size)
    S_cap, E_cap = superpixel_capacity(H, W, min_size)
    for _ in range(4):
        seeds = rng.random((k, 2)) * [H, W]
        yy, xx = np.mgrid[0:H, 0:W]
        lab = ((yy[..., None] - seeds[:, 0]) ** 2 + (xx[..., None] - seeds[:, 1]) ** 2).argmin(-1)
        noise = rng.random((H, W)) < 0.15
        lab[noise] = rng.integers(0, k, int(noise.sum()))
        out = _post_pass(lab, min_size)
        S = int(out.max()) + 1
        assert S <= S_cap and len(np.unique(out)) == S
        assert len(_components(out)[1]) == S                          # one component per final label
        assert 2 * len(_adjacent_pairs(out)) <= E_cap
