"""Step-by-step parity of the device CG, BiCGSTAB and GMRES solves with their fp64 references
(tests/test_{cg,bicgstab,gmres}_cpu.py), at the sizes where the solver kernels leave their
simplest paths:

- n = 1, 31, 33: one block, a partly masked warp (the GMRES warp loops mask their tail lanes and
  pad the basis column stride past n);
- n = 65,536: exactly kKrylovBlock blocks, so the last block adds the per-block partials in one
  pass (grid_sum, grid_sum_n in csrc/krylov.cuh);
- n = 65,537: one block more, with one live thread, so that loop wraps;
- n = BIG = 577 * 547: above the capped grid (kKrylovBlocksPerSm blocks per SM) times
  kKrylovBlock on a 148-SM B200, so every grid-stride loop, the warp-at-a-time ones of GMRES
  included, runs twice for part of the threads; n is not a multiple of 32.

A solve stopped after k steps (max_iter = k) returns the k-th iterate; it is compared with the
reference's k-th iterate to a relative tolerance T per solver.  A dropped term in a reduction
barely moves the converged count or the final residual, since the methods correct themselves,
but it moves the iterate at a fixed step by orders of magnitude more than rounding does.  The
unmarked tests prove each T on the CPU for every case the device tests use: (a) a second fp64
reference that differs only in summation order (the same reference on the permuted problem
P A P^T, with each row's entries reversed) stays within T / 10, and (b) the reference with the
last element dropped from one inner product (the first p.q of CG, the first (r^, v) of
BiCGSTAB, the first h2 of GMRES) moves x_k by at least 10 T, wherever the reference still runs
at step k (a solve that has converged by then has corrected the error away) and except where
drop_visible says why it cannot.  GMRES drops from h2, the second Gram-Schmidt pass: an error in
the first pass, h1, is measured and removed by the second, so x moves by rounding only."""
import functools
import os
import re

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from oracle import cpu
from test_bicgstab_cpu import bicgstab_reference, jacobi_dinv
from test_cg_cpu import pcg_reference
from test_gmres_cpu import gmres_reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BLOCK = 256          # kKrylovBlock in csrc/krylov.cuh: threads of a solver's streaming kernels
BLOCKS_PER_SM = 8    # kKrylovBlocksPerSm in csrc/krylov.cuh: the cap on their grid, per SM
B200_SMS = 148       # the SM count the sizes below are placed for

BIG_NX, BIG_NY = 577, 547
BIG = BIG_NX * BIG_NY
SIZES = (1, 31, 33, 65536, 65537, BIG)
GRID_WIDTH = {1: 1, 31: 6, 33: 6, 65536: 256, 65537: 257, BIG: BIG_NX}   # of the grid Laplacian

RTOL = 1e-10         # of the fixed-step solves: the big ones run every step, the small ones converge

# (matrix, jacobi, x0): each matrix with Jacobi off and on, each start with both; Jacobi runs on
# the row-scaled copy S A S, where diag(A) is not a multiple of I
VARIANTS = (("grid", False, "zero"), ("grid", True, "random"), ("irregular", False, "random"),
            ("irregular", True, "zero"))

# T, relative to ||x_ref||, per solver and step.  Each value sits between 10x the reordered
# reference's drift and 1/10 of a dropped element's effect (test_tolerance_holds_on_the_cpu).
# BiCGSTAB stops at k = 10: it amplifies rounding so fast that by k = 30 the reordered reference
# drifts by up to 6e-10 of ||x|| on the grid matrices, while a dropped element moves x by 3e-8.
TOL = {"cg": {1: 1e-13, 2: 1e-13, 5: 1e-13, 30: 1e-12, 100: 3e-13},
       "bicgstab": {1: 1e-13, 2: 1e-13, 5: 1e-13, 10: 1e-12}}
TOL_GMRES = 1e-13
# fp32: 10x the drift of a restatement that rounds to fp32 where the device stores a vector
TOL_F32 = 1e-4
F32_STEPS = (1, 2, 5)


def tol(solver, k):
    return TOL_GMRES if solver == "gmres" else TOL[solver][k]


def drop_visible(solver, n, k):
    """Whether (b) can hold.  GMRES minimises the residual over the Krylov space, and a wrong h2
    in the first step barely changes that space: on the big n the dropped element moves x_k by
    only 2e-15 to 1.4e-13 of ||x|| from k = m - 1 = 63 on, as little as rounding does.  Those
    comparisons still hold x to T, the rounding bound of (a)."""
    return not (solver == "gmres" and n == BIG and k > 2)


def restart_for(n):
    return 64 if n == BIG else 20


def steps(solver, name, n):
    """The k of the fixed-step comparisons.  The irregular matrices are strictly diagonally
    dominant, so their solves correct a dropped element within a few steps; the grid ones carry
    it to k = 100.  GMRES takes 1, 2, m - 1, m, m + 1, 2m + 3 for m = min(restart, n) on the grid
    matrices from n = 65,536 on; at n <= 33 the solve is within a few steps of converging at
    k = m - 1 .. m + 1, where a dropped element moves x by less than 100x rounding, and 2m + 3 is
    past convergence."""
    m = min(restart_for(n), n)
    if name == "irregular":
        return (1, 2) if solver == "gmres" else (1, 2, 5)
    if name == "split":
        return (2, m + 1) if solver == "gmres" else (5, 30)
    if solver != "gmres":
        return tuple(TOL[solver])
    ks = (1, 2, m - 1, m, m + 1, 2 * m + 3) if n > 33 else (1, 2, 2 * m + 3)
    return tuple(sorted({k for k in ks if k > 0}))


def krylov_blocks(n, sm_count):
    """krylov_grid in csrc/krylov.cuh"""
    return max(1, min(-(-n // BLOCK), BLOCKS_PER_SM * sm_count))


def check_boundaries(sm_count):
    """Each size lands on the side of the partials (256 blocks) and grid-stride (G * 256, G the
    grid cap) boundaries that the module docstring claims."""
    cap = BLOCKS_PER_SM * sm_count
    for n in (1, 31, 33):
        assert krylov_blocks(n, sm_count) == 1 and n % 32 != 0, n
    assert krylov_blocks(65536, sm_count) == BLOCK and 65536 <= cap * BLOCK
    assert krylov_blocks(65537, sm_count) == BLOCK + 1 and 65537 == BLOCK * BLOCK + 1 and 65537 <= cap * BLOCK
    assert krylov_blocks(BIG, sm_count) == cap > BLOCK
    assert BIG > cap * BLOCK and BIG % 32 != 0


# ---------------------------------------------------------------------------- matrices at any n

def csr(A, offset=np.int32):
    A = sp.csr_matrix(A)
    A.sum_duplicates()
    A.sort_indices()
    return A.indptr.astype(offset), A.indices.astype(np.int32), A.data.astype(np.float64)


def grid_laplacian(n, nx, convection=0.0):
    """The 5-point Laplacian (4, -1) on the first n points, row-major, of a grid nx wide: an
    nx x (n / nx) rectangle when nx divides n.  convection > 0 adds the upwind convection of
    test_bicgstab_cpu.convdiff along the grid rows (A[i,i] += c, A[i,i-1] -= c)."""
    i = np.arange(n, dtype=np.int64)
    c = i % nx
    cols = np.stack([i - nx, i - 1, i, i + 1, i + nx], axis=1)
    ok = np.stack([i >= nx, c > 0, np.ones(n, bool), (c < nx - 1) & (i + 1 < n), i + nx < n], axis=1)
    vals = np.broadcast_to(np.array([-1.0, -1.0 - convection, 4.0 + convection, -1.0, -1.0]), (n, 5))
    Ap = np.zeros(n + 1, np.int64)
    np.cumsum(ok.sum(axis=1), out=Ap[1:])
    return Ap.astype(np.int32), cols[ok].astype(np.int32), np.ascontiguousarray(vals[ok])


def irregular(n, symmetric, seed=7):
    """B + B^T + diag(1 + row sums of |B + B^T|) (symmetric: SPD), or B + diag(1 + row sums of
    |B|), for a random sparse B whose row lengths run from 0 to 400 (a Zipf tail), its values in
    [-1, 1] / sqrt(row length), so that a few long rows do not carry every inner product."""
    rng = np.random.default_rng(seed + n)
    lengths = np.minimum(rng.zipf(1.6, n) - 1, min(n, 400))
    rows = np.repeat(np.arange(n), lengths)
    cols = rng.integers(0, n, rows.size)
    vals = rng.uniform(-1.0, 1.0, rows.size) / np.sqrt(lengths[rows])
    B = sp.csr_matrix((vals, (rows, cols)), shape=(n, n))
    if symmetric:
        B = B + B.T
    d = 1.0 + np.asarray(abs(B).sum(axis=1)).ravel()
    return csr(B + sp.diags(d))


@functools.lru_cache(maxsize=None)
def matrix(solver, name, n, scaled):
    """fp64 CSR arrays (int32 offsets, sorted columns): the SPD pattern for CG, the
    nonsymmetric one for BiCGSTAB and GMRES; scaled: S A S with S in [1, 10]."""
    if name in ("grid", "split"):
        Ap, Aj, Ax = grid_laplacian(n, GRID_WIDTH[n], 0.0 if solver == "cg" else 1.0)
    else:
        Ap, Aj, Ax = irregular(n, solver == "cg")
    if scaled:
        s = np.random.default_rng(11).uniform(1.0, 10.0, n)
        rows = np.repeat(np.arange(n), np.diff(Ap))
        Ax = Ax * s[rows] * s[Aj]
    if name == "split":
        Ap, Aj, Ax = split_diagonals(Ap, Aj, Ax)
    return Ap, Aj, Ax


def split_diagonals(Ap, Aj, Ax, every=100):
    """Every `every`-th row's diagonal a stored as two entries, 0.375 a leading the row and
    0.625 a ending it: unsorted columns, and a diagonal that the SpMV and Jacobi must add."""
    n = Ap.shape[0] - 1
    rows = np.repeat(np.arange(n), np.diff(Ap))
    pick = (rows % every == every // 2) & (Aj == rows)
    r = np.concatenate([rows, rows[pick]])
    c = np.concatenate([Aj, Aj[pick]])
    v = np.concatenate([np.where(pick, 0.375 * Ax, Ax), 0.625 * Ax[pick]])
    pos = np.arange(rows.size) - Ap[rows]
    key = np.concatenate([np.where(pick, -1, pos), np.full(int(pick.sum()), rows.size)])
    order = np.lexsort((key, r))
    Ap2 = np.zeros(n + 1, np.int64)
    np.cumsum(np.bincount(r, minlength=n), out=Ap2[1:])
    return Ap2.astype(Ap.dtype), c[order].astype(np.int32), v[order]


@functools.lru_cache(maxsize=None)
def vectors(n, x0_kind):
    """b = A x_true is made per matrix; here x_true and x0 (zero or seeded in [-1, 1])"""
    x_true = np.random.default_rng(21).uniform(-1.0, 1.0, n)
    x0 = np.zeros(n) if x0_kind == "zero" else np.random.default_rng(22).uniform(-1.0, 1.0, n)
    return x_true, x0


@functools.lru_cache(maxsize=None)
def problem(solver, name, n, jacobi, x0_kind, dtype=np.float64):
    """(Ap, Aj, Ax, b, x0, dinv) in the value type (the reference reads the cast values
    exactly); dinv is the fp64 Jacobi diagonal or None"""
    Ap, Aj, Ax = matrix(solver, name, n, jacobi)
    x_true, x0 = vectors(n, x0_kind)
    Ax = Ax.astype(dtype)
    b = cpu.spmv_fp64(Ap, Aj, Ax, x_true).astype(dtype)
    return Ap, Aj, Ax, b, x0.astype(dtype), (jacobi_dinv(Ap, Aj, Ax) if jacobi else None)


def reference(solver, Ap, Aj, Ax, b, rtol, k, dinv, x0, trace=None):
    """(x, iterations, converged, breakdown) of the solver's reference, for max_iter = k"""
    if solver == "cg":
        return pcg_reference(Ap, Aj, Ax, b, rtol, k, dinv, x0, trace)
    if solver == "bicgstab":
        return bicgstab_reference(Ap, Aj, Ax, b, rtol, k, dinv, x0, trace)
    return gmres_reference(Ap, Aj, Ax, b, rtol, k, restart_for(Ap.shape[0] - 1), dinv, x0, trace=trace)


@functools.lru_cache(maxsize=None)
def ref_steps(solver, name, n, jacobi, x0_kind, k, dtype=np.float64):
    Ap, Aj, Ax, b, x0, dinv = problem(solver, name, n, jacobi, x0_kind, dtype)
    return reference(solver, Ap, Aj, Ax, b, RTOL, k, dinv, x0)


# ------------------------------------------------------- the second reference and the dropped term

def reordered(solver, Ap, Aj, Ax, b, rtol, k, dinv, x0, seed=5):
    """The reference on P A P^T, P b, P x0 with each row's entries in reverse order, mapped back:
    the same arithmetic with every dot product over a permuted order and every row summed in
    another order."""
    n = Ap.shape[0] - 1
    perm = np.random.default_rng(seed).permutation(n)
    inv = np.empty(n, np.int64)
    inv[perm] = np.arange(n)
    lengths = np.diff(Ap)[perm]
    Ap2 = np.zeros(n + 1, np.int64)
    np.cumsum(lengths, out=Ap2[1:])
    # entry t of new row i is entry (Ap[perm[i] + 1] - 1 - t) of old row perm[i]
    src = np.repeat(Ap[perm + 1].astype(np.int64) - 1 + Ap2[:-1], lengths) - np.arange(Ap2[-1])
    Aj2 = inv[Aj[src]].astype(np.int32)
    x, it, conv, brk = reference(solver, Ap2.astype(Ap.dtype), Aj2, Ax[src], b[perm], rtol, k,
                                 None if dinv is None else dinv[perm], x0[perm])
    return x[inv], it, conv, brk


def dropped(solver, Ap, Aj, Ax, b, k, dinv, x0, drop=True, store=None):
    """k steps of the reference's arithmetic (no stopping tests), with the last element dropped
    from the first p.q (CG), the first (r^, v) (BiCGSTAB) or the first h2 (GMRES) when drop is
    set.  store: a rounding applied where the device stores a vector in the value type (fp32),
    None for fp64.  With drop=False and store=None it returns the reference's bits."""
    n = Ap.shape[0] - 1
    st = (lambda v: v) if store is None else store

    def A(v):
        return st(cpu.spmv_fp64(Ap, Aj, Ax, v))

    def M(v):
        return v if dinv is None else st(dinv * v)

    def first(u, v, i):
        return u[:-1] @ v[:-1] if drop and i == 0 else u @ v

    x = np.array(x0, dtype=np.float64)
    if solver == "cg":
        r = st(b - A(x))
        z = M(r)
        p = z.copy()
        rho = r @ z
        for i in range(k):
            q = A(p)
            alpha = rho / first(p, q, i)
            x = st(x + st(alpha) * p)
            r = st(r - st(alpha) * q)
            z = M(r)
            rz = r @ z
            p = st(z + st(rz / rho) * p)
            rho = rz
        return x
    if solver == "bicgstab":
        r = st(b - A(x))
        rh = r.copy()
        rho = rh @ r
        for i in range(k):
            p = r.copy() if i == 0 else st(r + st(beta) * (p - st(omega) * v))  # noqa: F821
            ph = M(p)
            v = A(ph)
            alpha = rho / first(rh, v, i)
            s = st(r - st(alpha) * v)
            x = st(x + st(alpha) * ph)
            sh = M(s)
            t = A(sh)
            omega = (t @ s) / (t @ t)
            x = st(x + st(omega) * sh)
            r = st(s - st(omega) * t)
            rho_new = rh @ r
            beta = (rho_new / rho) * (alpha / omega)
            rho = rho_new
        return x
    m = min(restart_for(n), n)
    done = 0
    while done < k:
        cycle = min(m, k - done)
        r = st(b - A(x))
        V = np.zeros((m + 1, n))
        R = np.zeros((m, m))
        cs, sn, g = np.zeros(m), np.zeros(m), np.zeros(m + 1)
        g[0] = np.linalg.norm(r)
        V[0] = st(r / g[0])
        for j in range(cycle):
            w = A(M(V[j]))
            h1 = V[:j + 1] @ w
            w = st(w - V[:j + 1].T @ st(h1))
            h2 = V[:1, :-1] @ w[:-1] if drop and done == 0 and j == 0 else V[:j + 1] @ w
            w = st(w - V[:j + 1].T @ st(h2))
            hn = np.linalg.norm(w)
            col = h1 + h2
            for i in range(j):
                n0, n1 = col[i], col[i + 1]
                col[i] = cs[i] * n0 + sn[i] * n1
                col[i + 1] = -sn[i] * n0 + cs[i] * n1
            rr = np.hypot(col[j], hn)
            cs[j], sn[j] = col[j] / rr, hn / rr
            col[j] = rr
            R[j, :j + 1] = col
            g[j], g[j + 1] = cs[j] * g[j], -sn[j] * g[j]
            V[j + 1] = st(w * (1.0 / hn))
        y = g[:cycle].copy()
        for i in range(cycle - 1, 0, -1):
            y[i] /= R[i, i]
            y[:i] -= y[i] * R[i, :i]
        y[0] /= R[0, 0]
        x = st(x + M(y @ V[:cycle]))
        done += cycle
    return x


def rel(x, x_ref):
    return float(np.linalg.norm(np.asarray(x, np.float64) - x_ref) / np.linalg.norm(x_ref))


def f32(v):
    return v.astype(np.float32).astype(np.float64)


# --------------------------------------------------------------------------- the cases

SOLVERS = ("cg", "bicgstab", "gmres")


def _case(solver, name, n, jacobi, x0):
    return pytest.param(solver, name, n, jacobi, x0,
                        id=f"{solver}-{name}-n{n}-{'jacobi' if jacobi else 'plain'}-x0{x0}")


# every solver at every size, with every variant; on the big n also Jacobi CG and Jacobi GMRES on
# the grid matrix with split diagonals
PARITY = [_case(solver, name, n, jacobi, x0) for solver in SOLVERS for n in SIZES
          for name, jacobi, x0 in VARIANTS] + \
         [_case(solver, "split", BIG, True, "random") for solver in ("cg", "gmres")]
F32_CASES = [pytest.param(solver, n, id=f"{solver}-n{n}") for solver in SOLVERS for n in (65537, BIG)]
CONVERGED = [_case(solver, "irregular", BIG, jacobi, "zero") for solver in SOLVERS for jacobi in (False, True)]


# ------------------------------------------------------------------------- CPU: proofs of each T

def test_mirrored_constants_match_krylov_cuh():
    with open(os.path.join(ROOT, "spmv_samples_b200", "csrc", "krylov.cuh")) as f:
        src = f.read()
    found = dict(re.findall(r"constexpr\s+int\s+(kKrylov\w+)\s*=\s*(\d+)\s*;", src))
    assert int(found["kKrylovBlock"]) == BLOCK, found
    assert int(found["kKrylovBlocksPerSm"]) == BLOCKS_PER_SM, found


def test_sizes_sit_where_they_claim_on_a_b200():
    check_boundaries(B200_SMS)


def test_test_matrices_are_what_they_claim():
    Ap, Aj, Ax = matrix("cg", "grid", BIG, False)
    ref = sp.kron(sp.identity(BIG_NY), sp.diags([-1.0, 4.0, -1.0], [-1, 0, 1], (BIG_NX, BIG_NX))) \
        + sp.kron(sp.diags([-1.0, -1.0], [-1, 1], (BIG_NY, BIG_NY)), sp.identity(BIG_NX))
    assert abs(sp.csr_matrix((Ax, Aj, Ap), shape=(BIG, BIG)) - ref).max() == 0   # the 577 x 547 rectangle
    for n in (33, 65537):
        for solver in ("cg", "gmres"):
            Ap, Aj, Ax = matrix(solver, "irregular", n, False)
            A = sp.csr_matrix((Ax, Aj, Ap), shape=(n, n))
            d = A.diagonal()
            assert np.all(d - np.asarray(abs(A - sp.diags(d)).sum(axis=1)).ravel() >= 1.0 - 1e-9)
            assert (abs(A - A.T).max() == 0) == (solver == "cg")
            if n == 65537:
                lengths = np.diff(Ap)
                assert lengths.max() > 10 * np.median(lengths)          # uneven rows
    # split diagonals: the same matrix as an operator, ~1% of the rows with two diagonal entries
    for solver in ("cg", "gmres"):
        Ap, Aj, Ax = matrix(solver, "split", BIG, True)
        Ap0, Aj0, Ax0 = matrix(solver, "grid", BIG, True)
        rows = np.repeat(np.arange(BIG), np.diff(Ap))
        assert np.bincount(rows[Aj == rows], minlength=BIG).max() == 2
        assert 0.009 * BIG < Ap.shape[0] - 1 + Aj.size - Aj0.size - BIG < 0.011 * BIG + 1
        assert np.any(np.diff(Aj)[np.diff(rows) == 0] < 0)                # unsorted
        np.testing.assert_allclose(jacobi_dinv(Ap, Aj, Ax), jacobi_dinv(Ap0, Aj0, Ax0), rtol=1e-15)
        x = np.random.default_rng(1).uniform(-1.0, 1.0, BIG)
        np.testing.assert_allclose(cpu.spmv_fp64(Ap, Aj, Ax, x), cpu.spmv_fp64(Ap0, Aj0, Ax0, x),
                                   rtol=0, atol=1e-12 * np.abs(Ax0).max())


@pytest.mark.parametrize("solver", SOLVERS)
def test_restatement_reproduces_the_reference(solver):
    """dropped() without the drop is the reference's arithmetic, bit for bit, so (b) measures the
    dropped element alone"""
    for name, jacobi, x0 in VARIANTS:
        for n in (33, 65537) if name == "grid" else (33,):
            Ap, Aj, Ax, b, xs, dinv = problem(solver, name, n, jacobi, x0)
            k = min(steps(solver, name, n)[-1], 21)
            x, it, conv, _ = ref_steps(solver, name, n, jacobi, x0, k)
            if not conv:
                assert np.array_equal(dropped(solver, Ap, Aj, Ax, b, k, dinv, xs, drop=False), x), (name, n)


@pytest.mark.parametrize("solver,name,n,jacobi,x0", PARITY)
def test_tolerance_holds_on_the_cpu(solver, name, n, jacobi, x0):
    """(a) and (b) of the module docstring, at every k the device test uses"""
    Ap, Aj, Ax, b, xs, dinv = problem(solver, name, n, jacobi, x0)
    for k in steps(solver, name, n):
        T = tol(solver, k)
        x, it, conv, brk = ref_steps(solver, name, n, jacobi, x0, k)
        assert not brk and (conv or it == k), (k, it)
        x2, it2, conv2, _ = reordered(solver, Ap, Aj, Ax, b, RTOL, k, dinv, xs)
        assert (it2, conv2) == (it, conv), k
        assert rel(x2, x) <= T / 10, (k, rel(x2, x) / T)
        if not conv and drop_visible(solver, n, k):
            assert rel(dropped(solver, Ap, Aj, Ax, b, k, dinv, xs), x) >= 10 * T, k


@pytest.mark.parametrize("solver,n", F32_CASES)
def test_f32_tolerance_holds_on_the_cpu(solver, n):
    Ap, Aj, Ax, b, xs, dinv = problem(solver, "grid", n, False, "zero", np.float32)
    for k in F32_STEPS:
        x, it, conv, _ = ref_steps(solver, "grid", n, False, "zero", k, np.float32)
        assert it == k and not conv
        assert rel(dropped(solver, Ap, Aj, Ax, b, k, dinv, xs, drop=False, store=f32), x) <= TOL_F32 / 10, k


# --------------------------------------------------------------------------------- the device

@pytest.fixture(scope="module")
def device(built_lib):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    torch.cuda.set_device(0)
    yield torch.cuda.get_device_properties(0)
    from spmv_samples_b200 import spmv
    spmv.release_cache()


def run(solver, Ap, Aj, Ax, b, x0, k, kind, jacobi, rtol=RTOL, offset=np.int32):
    from spmv_samples_b200 import solve
    dev = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (Ap.astype(offset), Aj, Ax, b, x0)]
    n = Ap.shape[0] - 1
    extra = {"restart": restart_for(n)} if solver == "gmres" else {}
    return getattr(solve, solver)(*dev, rtol=rtol, max_iter=k, kind=kind, jacobi=jacobi, **extra)


def check_result(res, Ap, Aj, Ax, b, x_ref, it, conv, T, record_property, label):
    assert (res.iterations, res.converged, res.breakdown) == (it, conv, False), (label, res)
    x = res.x.cpu().numpy().astype(np.float64)
    ratio = rel(x, x_ref) / T
    record_property(label, f"{ratio:.3g}")
    assert ratio <= 1.0, (label, ratio)
    tr = float(np.linalg.norm(b.astype(np.float64) - cpu.spmv_fp64(Ap, Aj, Ax, x)))
    assert res.residual_norm == pytest.approx(tr, rel=1e-10), label
    assert res.b_norm == pytest.approx(float(np.linalg.norm(b.astype(np.float64))), rel=1e-12), label


@pytest.mark.gpu
def test_sizes_sit_where_they_claim_on_this_device(device):
    check_boundaries(device.multi_processor_count)


@pytest.mark.gpu
@pytest.mark.parametrize("solver,name,n,jacobi,x0", PARITY)
def test_fixed_steps_match_the_reference(device, record_property, solver, name, n, jacobi, x0):
    """max_iter = k: the k-th iterate, its count, residual and ||b||.  Kind auto with int32
    offsets everywhere; on the big n also merge and vector, and int64 offsets."""
    Ap, Aj, Ax, b, xs, dinv = problem(solver, name, n, jacobi, x0)
    combos = [(kind, off) for kind in ("auto", "merge", "vector") for off in (np.int32, np.int64)] \
        if n == BIG else [("auto", np.int32)]
    for k in steps(solver, name, n):
        x_ref, it, conv, _ = ref_steps(solver, name, n, jacobi, x0, k)
        for kind, off in combos:
            res = run(solver, Ap, Aj, Ax, b, xs, k, kind, jacobi, offset=off)
            check_result(res, Ap, Aj, Ax, b, x_ref, it, conv, tol(solver, k), record_property,
                         f"k{k}-{kind}-{np.dtype(off).name}")


@pytest.mark.gpu
@pytest.mark.parametrize("solver,n", F32_CASES)
def test_f32_steps_match_the_fp64_reference(device, record_property, solver, n):
    """fp32 values and vectors against the fp64 reference on the same (fp32) matrix and b.  This
    catches gross errors only: a dropped element moves x_k by about 1e-7 of ||x|| at these sizes,
    below the fp32 rounding."""
    Ap, Aj, Ax, b, xs, _ = problem(solver, "grid", n, False, "zero", np.float32)
    for k in F32_STEPS:
        x_ref, it, conv, _ = ref_steps(solver, "grid", n, False, "zero", k, np.float32)
        res = run(solver, Ap, Aj, Ax, b, xs, k, "auto", False)
        assert (res.iterations, res.converged, res.breakdown) == (it, conv, False), res
        ratio = rel(res.x.cpu().numpy(), x_ref) / TOL_F32
        record_property(f"k{k}", f"{ratio:.3g}")
        assert ratio <= 1.0, (k, ratio)


def deciding_norms(solver, Ap, Aj, Ax, b, x, trace):
    """every residual norm the reference compared with the tolerance"""
    if solver != "gmres":
        return trace
    return [e for cycle in trace for e in cycle] + [np.linalg.norm(b - cpu.spmv_fp64(Ap, Aj, Ax, x))]


@pytest.mark.gpu
@pytest.mark.parametrize("solver,name,n,jacobi,x0", CONVERGED)
def test_converged_count_equals_the_reference(device, solver, name, n, jacobi, x0):
    """rtol 1e-10 to convergence: the same iteration count as the reference, unless one of the
    reference's deciding residuals lies within 1e-6 (relative) of the tolerance"""
    Ap, Aj, Ax, b, xs, dinv = problem(solver, name, n, jacobi, x0)
    rtol = 1e-10
    trace = []
    x_ref, it, conv, brk = reference(solver, Ap, Aj, Ax, b, rtol, 10 * n, dinv, xs, trace)
    assert conv and not brk
    t = rtol * np.linalg.norm(b)
    if min(abs(v / t - 1.0) for v in deciding_norms(solver, Ap, Aj, Ax, b, x_ref, trace)) < 1e-6:
        pytest.skip("the reference decides within 1e-6 of the tolerance")
    res = run(solver, Ap, Aj, Ax, b, xs, None, "auto", jacobi, rtol)
    assert res.converged and not res.breakdown and res.iterations == it, (res, it)
    assert res.residual_norm <= 1.01 * t
