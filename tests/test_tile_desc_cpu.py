"""The tile descriptors of the persistent merge kernel (csrc/merge.cu, tile_desc_kernel), restated in
numpy from the merge-path coordinates of tests/reference_model.py.

row_end[r] = Ap[r+1] - sy(t) for the tile t in which row r's end item lies; the start mask has bit
q + shift of tile t set for every row end of the tile whose next row starts inside it (q < Z).  The
kernel finds t from the row's diagonal r + Ap[r+1]; the tile body reads row_end in place of Ap and
the mask in place of the flags its Ap scatter used to write, and takes b = 0 for a tile's first row.
These tests check that each of those readings is the same number as before."""
import numpy as np
import pytest

import reference_model as model
from oracle import generators as g

TILE = 128 * 8 - 4      # path items per tile of the persistent kernel (kTableBlock x kMergeIPT - 4)
SLOTS = TILE + 4


def lens_to_ap(lens, off=np.int32):
    Ap = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=Ap[1:])
    return Ap.astype(off)


def edge_shapes():
    """Row lengths that put row ends, row starts and empty rows on the tile edges."""
    rng = np.random.default_rng(17)
    return {
        # row 0 ends at diagonal T-1 / T / T+1: the last item of tile 0, the first and second of tile 1
        # (T-1: tile 1 starts exactly at row 1's first nonzero, Ap[sx] == sy)
        "row_end_at_T-1": [TILE - 1] + [3] * 700,
        "row_end_at_T": [TILE] + [3] * 700,
        "row_end_at_T+1": [TILE + 1] + [3] * 700,
        # empty-row runs longer than a CTA (128) and longer than a tile (a tile of row ends only)
        "empty_runs": [5] * 50 + [0] * 200 + [7] * 50 + [0] * 2500 + [3] * 300 + [0] * 129,
        # a hub row over hundreds of tiles, between short rows
        "hub_row": [2] * 100 + [300_000] + [1] * 2000,
        # nothing on an edge in particular; the last tile is partial
        "ragged": list(rng.integers(0, 40, 9000)),
    }


def matrices():
    out = {name: lens_to_ap(lens) for name, lens in edge_shapes().items()}
    out["rmat_s12"] = g.rmat(12, 16, 5)[0]
    out["rmat_s14_e8"] = g.rmat(14, 8, 3)[0]
    return out


def coords(Ap):
    """Row coordinate of the merge path at every tile boundary, from reference_model."""
    total = len(Ap) - 1 + int(Ap[-1])
    n_tiles = (total + TILE - 1) // TILE
    return np.array([model.merge_path_search(Ap, min(t * TILE, total))[0] for t in range(n_tiles + 1)],
                    dtype=np.int64)


def build_descriptors(Ap, cx):
    """What tile_desc_kernel writes: one thread per row, the tile found from the row's diagonal."""
    Ap = np.asarray(Ap, dtype=np.int64)
    n_rows, nnz = len(Ap) - 1, int(Ap[-1])
    total = n_rows + nnz
    n_tiles = len(cx) - 1
    r = np.arange(n_rows, dtype=np.int64)
    e = Ap[1:]
    t = (r + e) // TILE
    d0 = t * TILE
    d1 = np.minimum(d0 + TILE, total)
    sy = d0 - cx[t]
    ey = d1 - cx[t + 1]
    q = e - sy
    row_end = q.astype(np.uint16)
    bits = np.zeros((n_tiles, SLOTS), dtype=bool)
    starts = e < ey
    bits[t[starts], (q + (sy & 3))[starts]] = True
    return row_end, q, t, np.packbits(bits, axis=1, bitorder="little")


def scatter_flags(Ap, cx):
    """The byte flags of the Ap scatter in merge_tile_reg_body, tile by tile, and each row's tile."""
    Ap = np.asarray(Ap, dtype=np.int64)
    n_rows, nnz = len(Ap) - 1, int(Ap[-1])
    total = n_rows + nnz
    n_tiles = len(cx) - 1
    flags = np.zeros((n_tiles, SLOTS), dtype=bool)
    tile_of_row = np.full(n_rows, -1, dtype=np.int64)
    for tile in range(n_tiles):
        sx, ex = int(cx[tile]), int(cx[tile + 1])
        d0 = tile * TILE
        d1 = min(d0 + TILE, total)
        sy = d0 - sx
        Z = (d1 - ex) - sy
        q = Ap[sx + 1:ex + 1] - sy
        flags[tile, (q[q < Z] + (sy & 3))] = True
        tile_of_row[sx:ex] = tile
    return np.packbits(flags, axis=1, bitorder="little"), tile_of_row


@pytest.mark.parametrize("name", sorted(matrices()))
def test_descriptors_match_the_scatter_they_replace(name):
    Ap = matrices()[name]
    A64 = Ap.astype(np.int64)
    cx = coords(Ap)
    n_tiles = len(cx) - 1
    row_end, q, t, mask = build_descriptors(Ap, cx)
    flags, tile_of_row = scatter_flags(Ap, cx)
    # the tile found from the diagonal is the tile whose coordinates enclose the row
    assert np.array_equal(t, tile_of_row)
    # the merge path's invariant Ap[sx] <= sy: the first row of a tile starts at or before the tile
    sy = np.arange(n_tiles, dtype=np.int64) * TILE - cx[:-1]
    assert np.all(A64[cx[:-1]] <= sy)
    # every row end fits 16 bits: 0 <= q <= TILE
    assert q.min(initial=0) >= 0 and q.max(initial=0) <= TILE
    assert np.array_equal(row_end.astype(np.int64), q)
    # the mask is the scatter's flags, bit for bit
    assert mask.shape == (n_tiles, SLOTS // 8)
    assert np.array_equal(mask, flags)
    # the row-total loop and the carry: (b, q) and the last q of a tile as the Ap reads gave them
    for tile in range(n_tiles):
        sx, ex = int(cx[tile]), int(cx[tile + 1])
        for j in range(ex - sx):
            b_ap = max(int(A64[sx + j]) - int(sy[tile]), 0)
            b_desc = int(row_end[sx + j - 1]) if j else 0
            assert b_ap == b_desc, (name, tile, j)
        if ex > sx:
            assert int(A64[ex]) - int(sy[tile]) == int(row_end[ex - 1])
    if name == "row_end_at_T-1":
        assert A64[cx[1]] == sy[1]               # tile 1 starts exactly at its first row's first nonzero
    if name == "empty_runs":
        assert np.diff(cx).max() == TILE        # a tile of row ends only (more than 128 of them)
    if name == "hub_row":
        assert np.sum(np.diff(cx) == 0) >= 200   # hundreds of tiles without a row end
