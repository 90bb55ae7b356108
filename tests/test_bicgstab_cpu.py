"""CPU suite for the BiCGSTAB solve (spmvb200_bicgstab, spmv_samples_b200.solve.bicgstab): the
nonsymmetric test matrices, the numpy restatement of right-preconditioned BiCGSTAB that the GPU
tests compare with, pinned to scipy.sparse.linalg.bicgstab, and argument checks that need no
device."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import cpu
from oracle import generators as g
from test_cg_cpu import _valid_args


def convdiff(grid, c=1.0, dtype=np.float64, offset=np.int32):
    """lap2d(grid) with first-order upwind convection along the grid rows: A[i,i] += c and
    A[i,i-1] -= c where the west neighbour exists.  A nonsymmetric M-matrix."""
    Ap, Aj, Ax = g.lap2d(grid, np.float64, offset)
    rows = np.repeat(np.arange(Ap.shape[0] - 1), np.diff(Ap))
    Ax = Ax.copy()
    Ax[Aj == rows] += c
    Ax[Aj == rows - 1] -= c
    return Ap, Aj, Ax.astype(dtype)


def rmat_dominant(scale, ef=16, seed=3, dtype=np.float64, offset=np.int32):
    """R + diag(1 + sum_k |R_ik|) for the R-MAT matrix R of generators.rmat (the sum over its
    stored entries), duplicates summed and columns sorted, as scipy's R + diags(...) gives it.
    Its rows stay skewed (the longest holds 2552 entries at scale 14, seed 3); it is strictly
    diagonally dominant, so BiCGSTAB converges, in a few iterations with Jacobi."""
    Ap, Aj, Ax = g.rmat(scale, ef, seed, np.float64, np.int64)
    n = Ap.shape[0] - 1
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(Ap))
    diag = 1.0 + np.bincount(rows, weights=np.abs(Ax), minlength=n)
    keys, inv = np.unique(np.concatenate([rows * n + Aj, np.arange(n, dtype=np.int64) * (n + 1)]),
                          return_inverse=True)
    vals = np.bincount(inv, weights=np.concatenate([Ax, diag]))
    Ap2 = np.zeros(n + 1, np.int64)
    np.cumsum(np.bincount(keys // n, minlength=n), out=Ap2[1:])
    return Ap2.astype(offset), (keys % n).astype(np.int32), vals.astype(dtype)


def swap_pairs(pairs, dtype=np.float64, offset=np.int32):
    """Block-diagonal [[0, 1], [1, 0]]: with b = 1 on even indices, A b lives on odd ones, so
    (r^, v) = 0 in the first iteration."""
    n = 2 * pairs
    Ap = np.arange(n + 1).astype(offset)
    Aj = (np.arange(n) ^ 1).astype(np.int32)
    return Ap, Aj, np.ones(n, dtype)


def scaled_identity(n, d=4.0, dtype=np.float64, offset=np.int32):
    return np.arange(n + 1).astype(offset), np.arange(n, dtype=np.int32), np.full(n, d, dtype)


def jacobi_dinv(Ap, Aj, Ax):
    """1 / diag(A), duplicates added (what the device's Jacobi diagonal computes)."""
    n = Ap.shape[0] - 1
    rows = np.repeat(np.arange(n), np.diff(Ap))
    on = Aj == rows
    return 1.0 / np.bincount(rows[on], weights=Ax[on].astype(np.float64), minlength=n)


def bicgstab_reference(Ap, Aj, Ax, b, rtol, max_iter, dinv=None, x0=None, trace=None):
    """Right-preconditioned BiCGSTAB in fp64 on oracle.cpu.spmv_fp64, in the operation order of
    scipy.sparse.linalg.bicgstab, with the stopping rules of csrc/bicgstab.cu: converged when
    ||r|| <= rtol * ||b|| at the start or after an iteration, or ||s|| <= rtol * ||b|| at the
    half step (which counts as an iteration); breakdown at an exact zero or a non-finite value of
    rho, (r^, v), alpha, (t, t) or omega, or at omega == 0.  trace, a list, gets every ||r|| and
    ||s|| compared with the tolerance.  Returns (x, iterations, converged, breakdown)."""
    n = Ap.shape[0] - 1
    b = np.asarray(b, dtype=np.float64)
    x = np.zeros(n) if x0 is None else np.array(x0, dtype=np.float64)

    def A(v):
        return cpu.spmv_fp64(Ap, Aj, Ax, v)

    def M(v):
        return v if dinv is None else dinv * v

    def decides(v):
        if trace is not None:
            trace.append(np.linalg.norm(v))
        return np.linalg.norm(v) <= tol

    with np.errstate(all="ignore"):
        r = b - A(x)
        rh = r.copy()
        bnorm = np.linalg.norm(b)
        tol = rtol * bnorm
        if bnorm == 0:
            return np.zeros(n), 0, True, False
        if decides(r):
            return x, 0, True, False
        rho = rh @ r
        if rho == 0 or not np.isfinite(rho):
            return x, 0, False, True
        it = 0
        while it < max_iter:
            p = r.copy() if it == 0 else r + beta * (p - omega * v)  # noqa: F821 (set below)
            ph = M(p)
            v = A(ph)
            rv = rh @ v
            alpha = rho / rv
            if rv == 0 or not np.isfinite(rv) or not np.isfinite(alpha):
                return x, it, False, True
            s = r - alpha * v
            x = x + alpha * ph
            it += 1
            if decides(s):
                return x, it, True, False
            sh = M(s)
            t = A(sh)
            tt = t @ t
            omega = (t @ s) / tt
            if tt == 0 or not np.isfinite(omega):
                return x, it, False, True
            x = x + omega * sh
            r = s - omega * t
            if decides(r):
                return x, it, True, False
            rho_new = rh @ r
            if omega == 0 or rho_new == 0 or not np.isfinite(rho_new):
                return x, it, False, True
            beta = (rho_new / rho) * (alpha / omega)
            rho = rho_new
    return x, it, False, False


def scipy_bicgstab(Ap, Aj, Ax, b, rtol, max_iter, dinv=None):
    """scipy's solve and its iteration count on our terms: the callback count, plus one when it
    returned at the half step (then x is not the last iterate handed to the callback)."""
    sla = pytest.importorskip("scipy.sparse.linalg")
    sp = pytest.importorskip("scipy.sparse")
    n = Ap.shape[0] - 1
    A = sp.csr_matrix((Ax, Aj, Ap), shape=(n, n))
    seen = []
    xs, info = sla.bicgstab(A, b, rtol=rtol, atol=0.0, maxiter=max_iter,
                            M=None if dinv is None else sp.diags(dinv),
                            callback=lambda xk: seen.append(xk.copy()))
    half = not seen or not np.array_equal(xs, seen[-1])
    return xs, info, len(seen) + int(half)


@pytest.mark.parametrize("rtol", [1e-6, 1e-10])
@pytest.mark.parametrize("jacobi", [False, True], ids=["plain", "jacobi"])
@pytest.mark.parametrize("matrix", ["convdiff64", "rmat_dominant14"])
def test_reference_bicgstab_matches_scipy(matrix, jacobi, rtol):
    Ap, Aj, Ax = convdiff(64) if matrix == "convdiff64" else rmat_dominant(14)
    n = Ap.shape[0] - 1
    b = np.random.default_rng(1).uniform(-1.0, 1.0, n)
    dinv = jacobi_dinv(Ap, Aj, Ax) if jacobi else None
    x, it, conv, brk = bicgstab_reference(Ap, Aj, Ax, b, rtol, 4 * n, dinv)
    xs, info, it_s = scipy_bicgstab(Ap, Aj, Ax, b, rtol, 4 * n, dinv)
    assert conv and not brk and info == 0
    assert it == it_s, (it, it_s)
    np.testing.assert_allclose(x, xs, rtol=0, atol=1e-12 * np.abs(xs).max())


def test_test_matrices_are_what_they_claim():
    sp = pytest.importorskip("scipy.sparse")
    Ap, Aj, Ax = convdiff(16)
    A = sp.csr_matrix((Ax, Aj, Ap), shape=(256, 256))
    assert abs(A - A.T).max() == 1.0                                # nonsymmetric
    assert np.all(A.diagonal() == 5.0) and np.all(A.sum(axis=1) >= 0)  # M-matrix rows
    Ap, Aj, Ax = rmat_dominant(14)
    n = Ap.shape[0] - 1
    assert int(np.diff(Ap).max()) == 2552                          # the merge and long-row paths run
    rows = np.repeat(np.arange(n), np.diff(Ap))
    d = 1.0 / jacobi_dinv(Ap, Aj, Ax)
    off = np.bincount(rows[Aj != rows], weights=np.abs(Ax[Aj != rows]), minlength=n)
    assert np.all(d - off >= 1.0 - 1e-9)                           # strictly diagonally dominant
    # the scale-20 matrix of the table-plan test: 18.9 M merge-path items (rows + nonzeros)
    assert (1 << 20) + (1 << 20) * 17 == 18874368


def test_reference_bicgstab_breakdown_and_edges():
    # swap pairs: (r^, v) = 0 exactly, breakdown before x moves
    Ap, Aj, Ax = swap_pairs(8)
    b = np.where(np.arange(16) % 2 == 0, 1.0, 0.0)
    x, it, conv, brk = bicgstab_reference(Ap, Aj, Ax, b, 1e-8, 16)
    assert (it, conv, brk) == (0, False, True) and np.all(x == 0)
    # 4 I: alpha = 1/4 exactly (1 with Jacobi), s = 0, converged at the half step
    Ap, Aj, Ax = scaled_identity(16)
    b = np.random.default_rng(2).uniform(-1.0, 1.0, 16)
    for dinv in (None, jacobi_dinv(Ap, Aj, Ax)):
        x, it, conv, brk = bicgstab_reference(Ap, Aj, Ax, b, 1e-8, 16, dinv)
        assert (it, conv, brk) == (1, True, False)
        assert np.array_equal(x, b / 4)
    # b = 0, x0 the solution, max_iter = 0
    Ap, Aj, Ax = convdiff(8)
    x, it, conv, _ = bicgstab_reference(Ap, Aj, Ax, np.zeros(64), 1e-8, 64, x0=np.ones(64))
    assert (it, conv) == (0, True) and np.all(x == 0)
    x0 = np.arange(64, dtype=np.float64) % 5 - 2
    x, it, conv, _ = bicgstab_reference(Ap, Aj, Ax, cpu.spmv_fp64(Ap, Aj, Ax, x0), 1e-8, 64, x0=x0)
    assert (it, conv) == (0, True) and np.array_equal(x, x0)
    x, it, conv, brk = bicgstab_reference(Ap, Aj, Ax, np.ones(64), 1e-8, 0)
    assert (it, conv, brk) == (0, False, False)
    # NaN in b: breakdown before the first iteration
    bn = np.ones(64)
    bn[7] = np.nan
    x, it, conv, brk = bicgstab_reference(Ap, Aj, Ax, bn, 1e-8, 64)
    assert (it, conv, brk) == (0, False, True)


def test_bicgstab_argument_validation_needs_no_device(built_lib):
    """The statuses of spmvb200_cg's validation, case for case, before any CUDA call."""
    from spmv_samples_b200 import _lib
    L = built_lib
    out = _lib.CgOut()

    def status(**changes):
        a = _valid_args(_lib)
        for k, v in changes.items():
            setattr(a, k, v)
        return L.spmvb200_bicgstab(C.byref(a), C.byref(out))

    assert L.spmvb200_bicgstab(None, C.byref(out)) == 1
    assert L.spmvb200_bicgstab(C.byref(_valid_args(_lib)), None) == 1
    assert status(kind=6) == 1 and status(kind=-1) == 1
    assert status(flags=2) == 1 and status(flags=3) == 1
    for rtol in (0.0, -1e-6, float("nan")):
        assert status(rtol=rtol) == 1
    assert status(max_iter=-1) == 1
    for name in ("Ap", "Aj", "Ax", "b", "x"):
        assert status(**{name: None}) == 1, name
    assert status(x=0x4000) == 1
    assert status(n=-1) == 1 and status(nnz=-1) == 1
    assert status(Ap=0x1008) == 2
    assert status(value_bits=16) == 4
    out.iterations, out.converged = 7, 0
    assert status(n=0, nnz=0, Ap=None, Aj=None, Ax=None, b=None, x=None) == 0
    assert out.iterations == 0 and out.converged == 1 and out.breakdown == 0


def test_solve_bicgstab_checks_tensors_before_the_device():
    from spmv_samples_b200 import solve
    Ap, Aj, Ax = (torch.from_numpy(a) for a in convdiff(4))
    b = torch.ones(16, dtype=torch.float64)
    with pytest.raises(TypeError):
        solve.bicgstab(Ap, Aj, Ax, b.float())
    with pytest.raises(TypeError):
        solve.bicgstab(Ap, Aj.long(), Ax, b)
    with pytest.raises(TypeError):
        solve.bicgstab(Ap.short(), Aj, Ax, b)
    with pytest.raises(TypeError):
        solve.bicgstab(Ap, Aj, Ax, b, torch.zeros(16, dtype=torch.float32))
    with pytest.raises(ValueError, match="square"):
        Aj_wide = Aj.clone()
        Aj_wide[3] = 16
        solve.bicgstab(Ap, Aj_wide, Ax, b)
    with pytest.raises(ValueError, match="length"):
        solve.bicgstab(Ap, Aj, Ax, torch.ones(15, dtype=torch.float64))
    with pytest.raises(ValueError, match="length"):
        solve.bicgstab(Ap, Aj, Ax, b, torch.zeros(17, dtype=torch.float64))
    with pytest.raises(ValueError):
        solve.bicgstab(Ap, Aj, Ax, b, rtol=0.0)
    with pytest.raises(ValueError):
        solve.bicgstab(Ap, Aj, Ax, b, max_iter=-1)
    with pytest.raises(ValueError, match="different"):
        solve.bicgstab(Ap, Aj, Ax, b, b)
    with pytest.raises(ValueError, match="CUDA"):
        solve.bicgstab(Ap, Aj, Ax, b)
