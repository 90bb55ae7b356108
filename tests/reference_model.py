"""The original spmv-samples CPU code, restated in numpy.

The live comparisons in test_oracle.py and test_loader.py run against the original itself where
oracle/_ref has been built from its sources (`make -C oracle REFERENCE=<spmv-samples checkout>`).
Those sources are not part of this repository, so everywhere else the same comparisons run against
this restatement, which test_oracle.py first checks bit for bit against the golden vectors the
original produced (tests/golden/*.npz, *.mtx.npz).  Every function mirrors one `oracle.cpu.ref_*`:

  spmv, spmv_fp64, abs_scale, spmv_semiring   cpu_navie.hpp: per row, in CSR order, from the
                                              identity, each operation rounded in the stated type
  merge_path_search                           thread_search.cuh: CUB's MergePathSearch
  coo_to_csr, load_mtx                        load.hpp: LoadCoo (file order; an off-diagonal entry
                                              of a symmetric file followed by its mirror; values
                                              read as double, cast to float) + ToCsr (stable
                                              counting sort by row)
"""
import numpy as np


def _row_fold(Ap, terms, init, fold):
    """y[r] = fold(...fold(init, terms[Ap[r]])..., terms[Ap[r+1]-1]), k ascending."""
    Ap = np.asarray(Ap, dtype=np.int64)
    lens = np.diff(Ap)
    y = np.full(lens.size, init, dtype=terms.dtype)
    for k in range(int(lens.max(initial=0))):
        rows = np.nonzero(lens > k)[0]
        y[rows] = fold(y[rows], terms[Ap[rows] + k])
    return y


def spmv(Ap, Aj, Ax, x):
    """SpMV_cpu_navie: products and sums in the value type."""
    return _row_fold(Ap, Ax * np.asarray(x, dtype=Ax.dtype)[Aj], 0, np.add)


def spmv_fp64(Ap, Aj, Ax, x):
    return _row_fold(Ap, Ax.astype(np.float64) * np.asarray(x, dtype=np.float64)[Aj], 0, np.add)


def abs_scale(Ap, Aj, Ax, x):
    return _row_fold(Ap, np.abs(Ax.astype(np.float64) * np.asarray(x, dtype=np.float64)[Aj]), 0, np.add)


def spmv_semiring(Ap, Aj, Ax, x, semiring):
    xv = np.asarray(x, dtype=Ax.dtype)[Aj]
    if semiring == "min_plus":
        return _row_fold(Ap, Ax + xv, np.inf, np.minimum)
    if semiring == "max_plus":
        return _row_fold(Ap, Ax + xv, -np.inf, np.maximum)
    if semiring == "or_and":
        return _row_fold(Ap, ((Ax != 0) & (xv != 0)).astype(Ax.dtype), 0, np.maximum)
    raise ValueError(semiring)


def merge_path_search(Ap, diagonal):
    """(x, y) on the merge path of the row ends Ap[1:] and the nonzero indices: x is the first
    row r in [max(0, d - nnz), min(d, n_rows)] with Ap[r + 1] > d - r - 1, or the upper bound."""
    Ap = np.asarray(Ap, dtype=np.int64)
    n_rows, nnz = Ap.size - 1, int(Ap[-1])
    lo, hi = max(0, diagonal - nnz), min(diagonal, n_rows)
    f = Ap[1:] + np.arange(1, n_rows + 1)          # Ap[r + 1] + r + 1, non-decreasing
    x = int(np.searchsorted(f, diagonal, side="right"))
    x = min(hi, max(lo, x))
    return x, diagonal - x


def coo_to_csr(n_rows, rows, cols, vals):
    rows = np.asarray(rows, dtype=np.int64)
    order = np.argsort(rows, kind="stable")
    Ap = np.zeros(n_rows + 1, dtype=np.int32)
    Ap[1:] = np.cumsum(np.bincount(rows, minlength=n_rows))
    return Ap, np.asarray(cols, dtype=np.int32)[order], np.asarray(vals, dtype=np.float32)[order]


def load_mtx(filename):
    """Matrix Market coordinate file -> (n_rows, n_cols, Ap, Aj, Ax) with int32 offsets, fp32 values.
    Entries are read as a stream of tokens, so their line layout does not matter; lines after the
    announced number of entries are ignored."""
    with open(filename) as f:
        banner = f.readline().split()
        field, scheme = banner[3].lower(), banner[4].lower()
        assert banner[2].lower() == "coordinate" and scheme in ("general", "symmetric")
        line = f.readline()
        while not line.strip() or line.lstrip().startswith("%"):
            line = f.readline()
        n_rows, n_cols, entries = (int(t) for t in line.split())
        per = 2 if field == "pattern" else 3
        tok = f.read().split(maxsplit=per * entries)[:per * entries]
    assert len(tok) == per * entries
    r = np.array(tok[0::per], dtype=np.int64) - 1
    c = np.array(tok[1::per], dtype=np.int64) - 1
    v = np.ones(entries) if field == "pattern" else np.array([float(t) for t in tok[2::per]])
    if scheme == "symmetric":                     # (r, c, v) then (c, r, v) for r != c
        off = r != c
        pos = np.arange(entries) + np.cumsum(off) - off
        total = entries + int(off.sum())
        R, C, V = (np.empty(total, dtype=a.dtype) for a in (r, c, v))
        R[pos], C[pos], V[pos] = r, c, v
        R[pos[off] + 1], C[pos[off] + 1], V[pos[off] + 1] = c[off], r[off], v[off]
        r, c, v = R, C, V
    Ap, Aj, Ax = coo_to_csr(n_rows, r, c, v.astype(np.float32))
    return n_rows, n_cols, Ap, Aj, Ax


class _Restatement:
    """oracle.cpu's ref_* interface served by the functions above."""
    ref_spmv = staticmethod(spmv)
    ref_spmv_fp64 = staticmethod(spmv_fp64)
    ref_abs_scale = staticmethod(abs_scale)
    ref_spmv_semiring = staticmethod(spmv_semiring)
    ref_merge_path_search = staticmethod(merge_path_search)
    ref_load_mtx = staticmethod(load_mtx)

    @staticmethod
    def ref_coo_to_csr(n_rows, n_cols, rows, cols, vals):
        return coo_to_csr(n_rows, rows, cols, vals)

    @staticmethod
    def ref_spmv_mt(Ap, Aj, Ax, x, n_threads):
        """Row blocks on host threads: the oracle's run, which must equal the sequential loop."""
        from oracle import cpu
        return cpu.spmv_mt(Ap, Aj, Ax, x, n_threads)


def original():
    """The original's code: oracle.cpu's ref_* functions where oracle/_ref is built, else the
    restatement in this module."""
    from oracle import cpu
    return cpu if cpu.have_ref() else _Restatement
