"""CPU suite: pins oracle/ (the C restatement) against the reference.

1. the reference's only known-answer vector (merge_based/device_spmv.cuh:95-128);
2. golden vectors produced by the reference's own code (tests/golden/make_golden.py);
3. bit-for-bit comparison with the reference on fresh seeded inputs: live where oracle/_ref has
   been built from the reference's sources, elsewhere against their numpy restatement
   (tests/reference_model.py), itself pinned to the reference's golden vectors here.
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases, load_golden
from oracle import cpu, generators as g
import reference_model as model


def test_lattice_known_answer():
    d = load_golden("lattice3x3")
    assert d["Ap"].tolist() == [0, 2, 5, 7, 10, 14, 17, 19, 22, 24]
    y = cpu.spmv(d["Ap"], d["Aj"], d["Ax"], d["x"])
    assert y.tolist() == [2, 3, 2, 3, 4, 3, 2, 3, 2]


@pytest.mark.parametrize("name", golden_cases())
def test_oracle_matches_reference_golden(name):
    d = load_golden(name)
    Ap, Aj, Ax, x = d["Ap"], d["Aj"], d["Ax"], d["x"]
    assert np.array_equal(cpu.spmv(Ap, Aj, Ax, x), d["y_ref"])            # bit-exact
    assert np.array_equal(cpu.spmv_fp64(Ap, Aj, Ax, x), d["y_ref64"])
    assert np.array_equal(cpu.abs_scale(Ap, Aj, Ax, x), d["abs_ref"])
    for sr in cpu.SEMIRINGS:
        assert np.array_equal(cpu.spmv_semiring(Ap, Aj, Ax, x, sr), d[f"y_{sr}"])
        assert np.array_equal(cpu.spmv_semiring(Ap.astype(np.int64), Aj, Ax, x, sr), d[f"y_{sr}"])
    for tile in (2048, 896, 320):
        cx, cy = cpu.merge_tile_coords(Ap, tile)
        assert np.array_equal(np.stack([cx, cy], 1), d[f"coords_{tile}"])
    if "path_all" in d:
        n = Ap.shape[0] - 1 + int(Ap[-1])
        got = np.array([cpu.merge_path_search(Ap, k) for k in range(n + 1)], dtype=np.int64)
        assert np.array_equal(got, d["path_all"])
    # int64 offsets give the same answers
    Ap64 = Ap.astype(np.int64)
    assert np.array_equal(cpu.spmv(Ap64, Aj, Ax, x), d["y_ref"])
    cx64, _ = cpu.merge_tile_coords(Ap64, 2048)
    assert np.array_equal(cx64, d["coords_2048"][:, 0])


def test_oracle_mt_equals_sequential():
    Ap, Aj, Ax = g.ragged(5000, 700, 7.0, 21, heavy_len=9000)
    x = g.gen_x(5, 700)
    y = cpu.spmv(Ap, Aj, Ax, x)
    ymt, used = cpu.spmv_mt(Ap, Aj, Ax, x, 4)
    assert used >= 1 and np.array_equal(y, ymt)


def test_merge_path_properties():
    Ap, _, _ = g.ragged(2000, 100, 4.0, 17, heavy_len=7000)
    n_rows, nnz = Ap.shape[0] - 1, int(Ap[-1])
    cx, cy = cpu.merge_tile_coords(Ap, 512)
    assert cx[0] == 0 and cy[0] == 0 and cx[-1] == n_rows and cy[-1] == nnz
    assert np.all(np.diff(cx) >= 0) and np.all(np.diff(cy) >= 0)
    assert np.all((cx + cy)[:-1] == np.arange(len(cx) - 1) * 512)
    # a coordinate (i, j) on the path: all rows before i end at or before j; row i ends after j-1
    for i, j in zip(cx, cy):
        if i > 0:
            assert Ap[i] <= j
        if i < n_rows and j > 0:
            assert Ap[i + 1] > j - 1
    rb = cpu.row_split(Ap, 4)
    assert rb[0] == 0 and rb[-1] == n_rows and np.all(np.diff(rb) >= 0)


def test_coo_to_csr_stable_duplicates_kept():
    rows = np.array([2, 0, 2, 1, 0, 2, 2], dtype=np.int32)
    cols = np.array([5, 1, 3, 0, 1, 5, 0], dtype=np.int32)
    vals = np.arange(7, dtype=np.float32)
    Ap, Aj, Ax = cpu.coo_to_csr(4, rows, cols, vals)
    assert Ap.tolist() == [0, 2, 3, 7, 7]
    assert Aj.tolist() == [1, 1, 0, 5, 3, 5, 0]
    assert Ax.tolist() == [1, 4, 3, 0, 2, 5, 6]


def test_generators_shapes():
    Ap, Aj, Ax = g.lap2d(32)
    assert int(Ap[-1]) == 5 * 32 * 32 - 4 * 32 and Aj.max() == 32 * 32 - 1
    # each row: columns strictly ascending, diagonal 4, off-diagonals -1, row sums >= 0
    for r in (0, 31, 32, 500, 1023):
        c = Aj[Ap[r]:Ap[r + 1]]
        assert np.all(np.diff(c) > 0) and Ax[Ap[r]:Ap[r + 1]].sum() >= 0
    Ap, Aj, Ax = g.uniform_rows(128, 4096, 16, 3)
    assert np.all(np.diff(Ap) == 16)
    cols = Aj.reshape(128, 16)
    assert np.all(np.diff(cols, axis=1) > 0) and cols.max() < 4096 and cols.min() >= 0
    assert np.all(np.abs(Ax) <= 1)
    Ap, Aj, Ax = g.rmat(10, 16, 1)
    assert int(Ap[-1]) == 16 * 1024 and Aj.min() >= 0 and Aj.max() < 1024
    deg = np.diff(Ap)
    assert deg.max() > 8 * deg.mean()          # power law: a heavy head
    assert deg[0] == deg.max()                 # R-MAT's densest row is row 0
    # counter-based: a window of edges equals the same window of the full stream
    r_all, c_all = g.rmat_edges(10, 1, 0, 4096)
    r_win, c_win = g.rmat_edges(10, 1, 1000, 500)
    assert np.array_equal(r_all[1000:1500], r_win) and np.array_equal(c_all[1000:1500], c_win)


@pytest.mark.parametrize("name", golden_cases())
def test_numpy_restatement_matches_reference_golden(name):
    """tests/reference_model.py reproduces every golden vector of the reference bit for bit."""
    d = load_golden(name)
    Ap, Aj, Ax, x = d["Ap"], d["Aj"], d["Ax"], d["x"]
    assert np.array_equal(model.spmv(Ap, Aj, Ax, x), d["y_ref"])
    assert np.array_equal(model.spmv_fp64(Ap, Aj, Ax, x), d["y_ref64"])
    assert np.array_equal(model.abs_scale(Ap, Aj, Ax, x), d["abs_ref"])
    for sr in cpu.SEMIRINGS:
        assert np.array_equal(model.spmv_semiring(Ap, Aj, Ax, x, sr), d[f"y_{sr}"])
    total = Ap.shape[0] - 1 + int(Ap[-1])
    for tile in (2048, 896, 320):
        diags = np.minimum(np.arange(d[f"coords_{tile}"].shape[0]) * tile, total)
        got = np.array([model.merge_path_search(Ap, int(k)) for k in diags], dtype=np.int64)
        assert np.array_equal(got, d[f"coords_{tile}"])
    if "path_all" in d:
        got = np.array([model.merge_path_search(Ap, k) for k in range(total + 1)], dtype=np.int64)
        assert np.array_equal(got, d["path_all"])


ref = model.original()


class TestAgainstReferenceLive:
    """The oracle against the reference on fresh inputs: `ref` is the reference itself where
    oracle/_ref is built, else its restatement."""

    @pytest.mark.parametrize("seed", [1, 2, 3])
    def test_spmv_bit_exact(self, seed):
        Ap, Aj, Ax = g.ragged(3000, 900, 11.0, seed, heavy_len=4000)
        x = g.gen_x(seed, 900)
        assert np.array_equal(cpu.spmv(Ap, Aj, Ax, x), ref.ref_spmv(Ap, Aj, Ax, x))
        assert np.array_equal(cpu.spmv_fp64(Ap, Aj, Ax, x), ref.ref_spmv_fp64(Ap, Aj, Ax, x))
        assert np.array_equal(cpu.abs_scale(Ap, Aj, Ax, x), ref.ref_abs_scale(Ap, Aj, Ax, x))
        y, used = ref.ref_spmv_mt(Ap, Aj, Ax, x, 4)
        assert np.array_equal(y, ref.ref_spmv(Ap, Aj, Ax, x))
        for sr in cpu.SEMIRINGS:
            assert np.array_equal(cpu.spmv_semiring(Ap, Aj, Ax, x, sr),
                                  ref.ref_spmv_semiring(Ap, Aj, Ax, x, sr))

    def test_spmv_f64_and_o64(self):
        Ap, Aj, Ax = g.ragged(1000, 300, 20.0, 5, dtype=np.float64)
        x = g.gen_x(9, 300, np.float64)
        assert np.array_equal(cpu.spmv(Ap, Aj, Ax, x), ref.ref_spmv(Ap, Aj, Ax, x))
        Ap32, Aj, Ax = g.rmat(9, 16, 4)
        x = g.gen_x(2, 512)
        Ap64 = Ap32.astype(np.int64)
        assert np.array_equal(cpu.spmv(Ap64, Aj, Ax, x), ref.ref_spmv(Ap64, Aj, Ax, x))

    def test_search_every_diagonal(self):
        Ap, _, _ = g.ragged(400, 50, 3.0, 8, heavy_len=900)
        total = Ap.shape[0] - 1 + int(Ap[-1])
        for d in range(total + 1):
            assert cpu.merge_path_search(Ap, d) == ref.ref_merge_path_search(Ap, d)
        Ap64 = Ap.astype(np.int64)
        for d in range(0, total + 1, 7):
            assert cpu.merge_path_search(Ap64, d) == ref.ref_merge_path_search(Ap64, d)

    def test_coo_to_csr(self):
        rng = np.random.default_rng(0)
        rows = rng.integers(0, 50, 2000).astype(np.int32)
        cols = rng.integers(0, 70, 2000).astype(np.int32)
        vals = rng.uniform(-1, 1, 2000).astype(np.float32)
        a = cpu.coo_to_csr(50, rows, cols, vals)
        b = ref.ref_coo_to_csr(50, 70, rows, cols, vals)
        for u, v in zip(a, b):
            assert np.array_equal(u, v)

    def test_loader_fixtures_match_reference(self):
        for f in ("general_real.mtx", "symmetric_pattern.mtx", "symmetric_integer.mtx"):
            n_rows, n_cols, Ap, Aj, Ax = ref.ref_load_mtx(os.path.join(GOLDEN, f))
            d = np.load(os.path.join(GOLDEN, f + ".npz"))
            assert n_rows == int(d["n_rows"]) and n_cols == int(d["n_cols"])
            assert np.array_equal(Ap, d["Ap"]) and np.array_equal(Aj, d["Aj"])
            assert np.array_equal(Ax, d["Ax"])
