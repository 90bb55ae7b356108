"""CPU suite: include/load.hpp (the product's Matrix Market loader + COO->CSR) against the
reference's loader.  The expected CSR arrays in tests/golden/*.mtx.npz were produced by the
reference's own LoadCoo + ToCsr (tests/golden/make_golden.py).  On freshly written files the
comparison is made with the reference loader where oracle/_ref is built, else with its numpy
restatement (tests/reference_model.py, pinned to those golden arrays in test_oracle.py)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from oracle import cpu
import reference_model as model

SHIM_SRC = os.path.join(ROOT, "tests", "cxx", "loader_shim.cpp")
SHIM_SO = os.path.join(ROOT, "tests", "cxx", "libloader_shim.so")


@pytest.fixture(scope="module")
def shim():
    if (not os.path.exists(SHIM_SO) or os.path.getmtime(SHIM_SO) < max(
            os.path.getmtime(SHIM_SRC), os.path.getmtime(os.path.join(ROOT, "include", "load.hpp")))):
        gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.run([gxx, "-std=c++17", "-O2", "-fPIC", "-shared", "-fvisibility=hidden",
                        "-I" + os.path.join(ROOT, "include"), SHIM_SRC, "-o", SHIM_SO], check=True)
    return C.CDLL(SHIM_SO)


def load(shim, path, wide=False):
    h = C.c_void_p()
    n_rows, n_cols, nnz = C.c_int64(), C.c_int64(), C.c_int64()
    scheme = C.c_int()
    err = C.create_string_buffer(256)
    fn = shim.shim_load_o64_f64 if wide else shim.shim_load_o32_f32
    rc = fn(path.encode(), C.byref(h), C.byref(n_rows), C.byref(n_cols), C.byref(nnz),
            C.byref(scheme), err, 256)
    if rc != 0:
        return rc, err.value.decode()
    Ap = np.empty(n_rows.value + 1, dtype=np.int64 if wide else np.int32)
    Aj = np.empty(nnz.value, dtype=np.int32)
    Ax = np.empty(nnz.value, dtype=np.float64 if wide else np.float32)
    (shim.shim_copy_o64_f64 if wide else shim.shim_copy_o32_f32)(
        h, Ap.ctypes.data_as(C.c_void_p), Aj.ctypes.data_as(C.c_void_p), Ax.ctypes.data_as(C.c_void_p))
    return 0, (n_rows.value, n_cols.value, Ap, Aj, Ax)


@pytest.mark.parametrize("fname", ["general_real.mtx", "symmetric_pattern.mtx", "symmetric_integer.mtx"])
def test_fixture_matches_reference_loader(shim, fname):
    rc, out = load(shim, os.path.join(GOLDEN, fname))
    assert rc == 0, out
    n_rows, n_cols, Ap, Aj, Ax = out
    d = np.load(os.path.join(GOLDEN, fname + ".npz"))
    assert n_rows == int(d["n_rows"]) and n_cols == int(d["n_cols"])
    assert np.array_equal(Ap, d["Ap"]) and np.array_equal(Aj, d["Aj"]) and np.array_equal(Ax, d["Ax"])
    # 64-bit offsets / fp64 values: same structure
    rc, out = load(shim, os.path.join(GOLDEN, fname), wide=True)
    assert rc == 0 and np.array_equal(out[2], d["Ap"]) and np.array_equal(out[3], d["Aj"])


def _write_random_mtx(path, n_rows, n_cols, nnz, seed, field="real", scheme="general"):
    rng = np.random.default_rng(seed)
    r = rng.integers(1, n_rows + 1, nnz)
    c = rng.integers(1, n_cols + 1, nnz)
    if scheme != "general":
        r, c = np.maximum(r, c), np.minimum(r, c)   # lower triangle
        if scheme == "skew-symmetric":
            keep = r != c
            r, c = r[keep], c[keep]
    v = rng.uniform(-3, 3, r.size)
    with open(path, "w") as f:
        f.write(f"%%MatrixMarket matrix coordinate {field} {scheme}\n% generated\n%\n")
        f.write(f"{n_rows} {n_cols} {r.size}\n")
        for i in range(r.size):
            if field == "pattern":
                f.write(f"{r[i]} {c[i]}\n")
            elif field == "integer":
                f.write(f"{r[i]}\t{c[i]}  {int(v[i])}\n")
            else:
                f.write(f" {r[i]} {c[i]} {v[i]:.17g}\n")
    return r - 1, c - 1, v


@pytest.mark.parametrize("field,scheme", [("real", "general"), ("pattern", "general"),
                                          ("integer", "general"), ("real", "symmetric"),
                                          ("pattern", "symmetric")])
def test_random_files_match_reference_loader_live(shim, tmp_path, field, scheme):
    path = str(tmp_path / "m.mtx")
    _write_random_mtx(path, 300, 300 if scheme != "general" else 217, 5000, 5, field, scheme)
    rc, out = load(shim, path)
    assert rc == 0, out
    n_rows, n_cols, Ap, Aj, Ax = out
    rn, rc_, rAp, rAj, rAx = model.original().ref_load_mtx(path)
    assert (n_rows, n_cols) == (rn, rc_)
    assert np.array_equal(Ap, rAp) and np.array_equal(Aj, rAj) and np.array_equal(Ax, rAx)


def test_tocsr_is_the_oracles_counting_sort(shim, tmp_path):
    path = str(tmp_path / "m.mtx")
    r, c, v = _write_random_mtx(path, 100, 80, 3000, 9)
    rc, out = load(shim, path)
    assert rc == 0
    _, _, Ap, Aj, Ax = out
    eAp, eAj, eAx = cpu.coo_to_csr(100, r, c, v.astype(np.float32))
    assert np.array_equal(Ap, eAp) and np.array_equal(Aj, eAj) and np.array_equal(Ax, eAx)


def test_skew_and_hermitian_are_expanded(shim, tmp_path):
    """Deliberate deviation (SURVEY.md A.3): the reference loads these as half a matrix."""
    p = str(tmp_path / "skew.mtx")
    open(p, "w").write("%%MatrixMarket matrix coordinate real skew-symmetric\n3 3 2\n2 1 5\n3 2 -2\n")
    rc, (n, m, Ap, Aj, Ax) = load(shim, p)
    dense = np.zeros((3, 3))
    for r in range(3):
        for k in range(Ap[r], Ap[r + 1]):
            dense[r, Aj[k]] += Ax[k]
    assert np.array_equal(dense, np.array([[0, -5, 0], [5, 0, 2], [0, -2, 0]]))
    p = str(tmp_path / "herm.mtx")
    open(p, "w").write("%%MatrixMarket matrix coordinate real hermitian\n2 2 2\n1 1 1\n2 1 3\n")
    rc, (n, m, Ap, Aj, Ax) = load(shim, p)
    assert Ap.tolist() == [0, 2, 3] and Aj.tolist() == [0, 1, 0] and Ax.tolist() == [1, 3, 3]


def test_error_behaviour(shim, tmp_path):
    assert load(shim, str(tmp_path / "missing.mtx"))[0] == 11          # MM_COULD_NOT_READ_FILE
    p = str(tmp_path / "a.mtx")
    open(p, "w").write("%%MatrixMarket matrix array real general\n2 2\n1\n2\n3\n4\n")
    assert load(shim, p)[0] == 13                                        # not a sparse matrix
    open(p, "w").write("%%NotMatrixMarket matrix coordinate real general\n1 1 0\n")
    assert load(shim, p)[0] == 14                                        # no header
    open(p, "w").write("%%MatrixMarket matrix coordinate complex general\n1 1 1\n1 1 1 0\n")
    assert load(shim, p)[0] == 15                                        # unsupported field
    open(p, "w").write("%%MatrixMarket matrix coordinate real general\n2 2 1\n0 1 1.0\n")
    rc, msg = load(shim, p)
    assert rc == 100 and "zero-indexed" in msg                           # reference's exception text
    open(p, "w").write("%%MatrixMarket matrix coordinate real general\n2 2 3\n1 1 1.0\n")
    rc, msg = load(shim, p)
    assert rc == 100 and "Could not read weighted edge" in msg
    open(p, "w").write("%%MatrixMarket matrix coordinate real general\n3000000000 2 1\n1 1 1.0\n")
    rc, msg = load(shim, p)
    assert rc == 100 and "vertex_t overflow" in msg


def test_blank_lines_and_case_insensitive_banner(shim, tmp_path):
    p = str(tmp_path / "b.mtx")
    open(p, "w").write("%%MatrixMarket MATRIX Coordinate Real GENERAL\n%c\n\n2 3 2\n\n1 3 1e0\n2 1 -2.5E+0\n")
    rc, (n, m, Ap, Aj, Ax) = load(shim, p)
    assert (n, m) == (2, 3) and Ap.tolist() == [0, 1, 2] and Aj.tolist() == [2, 0] and Ax.tolist() == [1.0, -2.5]


def _write_big_mtx(path, n, nnz, seed, field="real", scheme="general", fmt="%d %d %.17g"):
    rng = np.random.default_rng(seed)
    r = rng.integers(1, n + 1, nnz)
    c = rng.integers(1, n + 1, nnz)
    if scheme != "general":
        r, c = np.maximum(r, c), np.minimum(r, c)
    v = rng.uniform(-3, 3, nnz) * 10.0 ** rng.integers(-30, 30, nnz)   # exercises the strtod fallback too
    with open(path, "w") as f:
        f.write(f"%%MatrixMarket matrix coordinate {field} {scheme}\n% big\n{n} {n} {nnz}\n")
        if field == "pattern":
            np.savetxt(f, np.column_stack([r, c]), fmt="%d %d")
        else:
            np.savetxt(f, np.column_stack([r, c, v]), fmt=fmt)


@pytest.mark.parametrize("threads", ["1", "3", "8"])
@pytest.mark.parametrize("field,scheme", [("real", "general"), ("real", "symmetric"), ("pattern", "general")])
def test_threaded_paths_match_reference_loader(shim, tmp_path, monkeypatch, field, scheme, threads):
    """Files large enough for the line-parallel parser and the threaded ToCsr (>= 256 KB, >= 2^17
    entries), with 1, 3 and 8 threads: the arrays must be the reference loader's, bit for bit."""
    monkeypatch.setenv("SPMV_LOADER_THREADS", threads)
    path = str(tmp_path / "big.mtx")
    _write_big_mtx(path, 5000, 150_000, 3, field, scheme)
    rc, out = load(shim, path)
    assert rc == 0, out
    n_rows, n_cols, Ap, Aj, Ax = out
    rn, rc_, rAp, rAj, rAx = model.original().ref_load_mtx(path)
    assert (n_rows, n_cols) == (rn, rc_)
    assert np.array_equal(Ap, rAp) and np.array_equal(Aj, rAj) and np.array_equal(Ax, rAx)
    # 64-bit offsets, fp64 values through the same paths
    rc, out = load(shim, path, wide=True)
    assert rc == 0 and np.array_equal(out[2], rAp) and np.array_equal(out[3], rAj)
    assert np.array_equal(out[4].astype(np.float32), rAx)


def test_unusual_layouts_fall_back_to_the_tokenizer(shim, tmp_path, monkeypatch):
    """Two entries on one line, an entry split over two lines, trailing lines after the last
    entry: the per-line parser declines and the sequential tokenizer gives the reference's result."""
    monkeypatch.setenv("SPMV_LOADER_THREADS", "4")
    rng = np.random.default_rng(8)
    n, nnz = 3000, 40_000
    r, c, v = rng.integers(1, n + 1, nnz), rng.integers(1, n + 1, nnz), rng.uniform(-1, 1, nnz)
    path = str(tmp_path / "odd.mtx")
    with open(path, "w") as f:
        f.write(f"%%MatrixMarket matrix coordinate real general\n{n} {n} {nnz}\n")
        i = 0
        while i < nnz:
            if i % 7 == 0 and i + 1 < nnz:      # two entries on one line
                f.write(f"{r[i]} {c[i]} {v[i]:.9g}   {r[i+1]} {c[i+1]} {v[i+1]:.9g}\n")
                i += 2
            elif i % 11 == 0:                    # one entry over two lines
                f.write(f"{r[i]} {c[i]}\n   {v[i]:.9g}\n")
                i += 1
            else:
                f.write(f"{r[i]} {c[i]} {v[i]:.9g}\n")
                i += 1
        f.write("1 1 99\n2 2 99\n")             # beyond the announced count: ignored
    rc, out = load(shim, path)
    assert rc == 0, out
    rn, rc_, rAp, rAj, rAx = model.original().ref_load_mtx(path)
    assert np.array_equal(out[2], rAp) and np.array_equal(out[3], rAj) and np.array_equal(out[4], rAx)


def test_errors_come_from_one_place_whatever_the_size(shim, tmp_path, monkeypatch):
    """A zero index deep inside a large file: same exception text as in a small one."""
    monkeypatch.setenv("SPMV_LOADER_THREADS", "4")
    path = str(tmp_path / "zero.mtx")
    with open(path, "w") as f:
        f.write("%%MatrixMarket matrix coordinate real general\n1000 1000 60000\n")
        for i in range(60000):
            f.write(f"{1 + i % 1000} {0 if i == 43210 else 1 + (7 * i) % 1000} 1.5\n")
    rc, msg = load(shim, path)
    assert rc == 100 and "zero-indexed" in msg
    with open(path, "w") as f:                    # short file
        f.write("%%MatrixMarket matrix coordinate real general\n1000 1000 60000\n")
        for i in range(59000):
            f.write(f"{1 + i % 1000} {1 + (7 * i) % 1000} 1.5\n")
    rc, msg = load(shim, path)
    assert rc == 100 and "Could not read weighted edge" in msg


@pytest.mark.parametrize("threads", ["1", "4"])
def test_out_of_range_indices_are_rejected(shim, tmp_path, monkeypatch, threads):
    """An index beyond the header's dimensions is an error in every parse path (the reference
    stores it unchecked, load.hpp:330-331, and its ToCsr then indexes past row_offsets)."""
    monkeypatch.setenv("SPMV_LOADER_THREADS", threads)
    p = str(tmp_path / "oob.mtx")
    open(p, "w").write("%%MatrixMarket matrix coordinate real general\n3 3 3\n1 1 1.0\n2 7 2.0\n3 3 3.0\n")
    rc, msg = load(shim, p)
    assert rc == 100 and "column index exceeds" in msg
    open(p, "w").write("%%MatrixMarket matrix coordinate pattern symmetric\n3 3 2\n1 1\n4 2\n")
    rc, msg = load(shim, p)
    assert rc == 100 and "row index exceeds" in msg
    # deep inside a file large enough for the threaded by-line path and the threaded ToCsr
    with open(p, "w") as f:
        f.write("%%MatrixMarket matrix coordinate real general\n1000 1000 200000\n")
        for i in range(200000):
            f.write(f"{1001 if i == 123456 else 1 + i % 1000} {1 + (7 * i) % 1000} 1.5\n")
    rc, msg = load(shim, p)
    assert rc == 100 and "row index exceeds" in msg
    with open(p, "w") as f:
        f.write("%%MatrixMarket matrix coordinate real general\n1000 1000 200000\n")
        for i in range(200000):
            f.write(f"{1 + i % 1000} {1001 if i == 199999 else 1 + (7 * i) % 1000} 1.5\n")
    rc, msg = load(shim, p)
    assert rc == 100 and "column index exceeds" in msg
    # the largest legal indices still load
    open(p, "w").write("%%MatrixMarket matrix coordinate real general\n3 4 1\n3 4 2.5\n")
    rc, out = load(shim, p)
    assert rc == 0 and out[2].tolist() == [0, 0, 0, 1] and out[3].tolist() == [3]
