"""CPU: the host half of the ragged resize (ops._ragged_plan): per-image records, table offsets and horizontal-pass rows,
derived from the shapes alone, laid out as include/gnc.h's gnc_resize_image."""
import numpy as np


def _plan(shapes, oh, ow):
    from graphnet_classifier_b200 import ops
    return ops._ragged_plan([s[0] for s in shapes], [s[1] for s in shapes], oh, ow)


def test_record_layout_matches_the_header():
    from graphnet_classifier_b200 import _lib
    d = np.dtype(_lib.GncResizeImage)
    assert d.itemsize == 56
    assert [d.fields[k][1] for k in ("src", "pitch", "tmp_row", "tab_x", "tab_y", "height", "width", "ksize_x", "ksize_y")] \
        == [0, 8, 16, 24, 32, 40, 44, 48, 52]


def test_taps_equal_the_library(libgnc):
    sizes = list(range(1, 700)) + [999, 1000, 1001, 2999, 3000, 4000, 12000]
    for out in (1, 2, 3, 24, 127, 128, 129, 333, 512):
        rec, _, _, _ = _plan([(s, s) for s in sizes], out, out)
        want = [0 if s == out else libgnc.gnc_resize_bicubic_ksize(s, out) for s in sizes]
        assert list(rec["ksize_x"]) == want and list(rec["ksize_y"]) == want, out


def test_offsets_tile_the_workspace_and_rows_find_their_image():
    rng = np.random.default_rng(0)
    oh, ow = 96, 128
    shapes = [(int(h), int(w)) for h, w in rng.integers(1, 900, (200, 2))]
    shapes += [(oh, ow), (oh, 7), (5, ow), (1, 1), (oh, ow)]
    rng.shuffle(shapes)
    rec, n_tables, h_rows, max_w = _plan(shapes, oh, ow)
    pos = 0
    for r, (h, w) in zip(rec, shapes):
        assert (r["height"], r["width"]) == (h, w)
        assert (r["ksize_x"] == 0) == (w == ow) and (r["ksize_y"] == 0) == (h == oh)
        assert r["tab_x"] == pos                          # x table, then y table, image after image, no gaps
        pos += ow * (2 + r["ksize_x"]) if r["ksize_x"] else 0
        assert r["tab_y"] == pos
        pos += oh * (2 + r["ksize_y"]) if r["ksize_y"] else 0
    assert pos == n_tables
    changed = [s for s in shapes if s[1] != ow]
    assert h_rows == sum(h for h, _ in changed) and max_w == max(w for _, w in changed)
    assert list(rec["tmp_row"]) == list(np.cumsum([0] + [h if w != ow else 0 for h, w in shapes])[:-1])
    # the horizontal kernel's search: a row belongs to the last image whose tmp_row is <= the row
    for row in range(h_rows):
        i = int(np.searchsorted(rec["tmp_row"], row, side="right")) - 1
        assert rec["ksize_x"][i] != 0 and 0 <= row - rec["tmp_row"][i] < rec["height"][i], row


def test_nothing_to_filter():
    rec, n_tables, h_rows, max_w = _plan([(64, 64), (64, 64)], 64, 64)
    assert n_tables == 0 and h_rows == 0 and max_w == 0
    assert not rec["ksize_x"].any() and not rec["ksize_y"].any()
