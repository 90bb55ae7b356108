"""CPU suite for the conjugate-gradient solve (spmvb200_cg, spmv_samples_b200.solve): argument
checks that need no device, and the numpy restatement of preconditioned CG that the GPU tests
compare with, pinned to scipy.sparse.linalg.cg."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import cpu
from oracle import generators as g


def pcg_reference(Ap, Aj, Ax, b, rtol, max_iter, dinv=None, x0=None, trace=None):
    """Preconditioned CG (Hestenes-Stiefel) in fp64 on oracle.cpu.spmv_fp64, with the stopping
    rules of csrc/cg.cu: converged when ||r|| <= rtol * ||b|| after an update (or at the start),
    breakdown when p.q <= 0.  trace, a list, gets every ||r|| compared with the tolerance.
    Returns (x, iterations, converged, breakdown)."""
    n = Ap.shape[0] - 1
    b = np.asarray(b, dtype=np.float64)
    x = np.zeros(n) if x0 is None else np.array(x0, dtype=np.float64)
    r = b - cpu.spmv_fp64(Ap, Aj, Ax, x)
    z = r if dinv is None else dinv * r
    p = z.copy()
    rho = r @ z
    tol = rtol * np.linalg.norm(b)
    if np.linalg.norm(b) == 0:
        return np.zeros(n), 0, True, False
    if trace is not None:
        trace.append(np.linalg.norm(r))
    if np.linalg.norm(r) <= tol:
        return x, 0, True, False
    it = 0
    while it < max_iter:
        q = cpu.spmv_fp64(Ap, Aj, Ax, p)
        pq = p @ q
        if not (pq > 0 and np.isfinite(pq)):
            return x, it, False, True
        alpha = rho / pq
        x = x + alpha * p
        r = r - alpha * q
        it += 1
        if trace is not None:
            trace.append(np.linalg.norm(r))
        if np.linalg.norm(r) <= tol:
            return x, it, True, False
        z = r if dinv is None else dinv * r
        rz = r @ z
        p = z + (rz / rho) * p
        rho = rz
    return x, it, False, False


def scaled(Ap, Aj, Ax, s):
    """S A S for the diagonal S = diag(s): symmetric and SPD when A is."""
    rows = np.repeat(np.arange(Ap.shape[0] - 1), np.diff(Ap))
    return Ap, Aj, (Ax.astype(np.float64) * s[rows] * s[Aj]).astype(Ax.dtype)


def test_reference_pcg_matches_scipy():
    sla = pytest.importorskip("scipy.sparse.linalg")
    sp = pytest.importorskip("scipy.sparse")
    Ap, Aj, Ax = g.lap2d(32, np.float64)
    n = Ap.shape[0] - 1
    s = np.random.default_rng(3).uniform(1.0, 10.0, n)
    b = np.random.default_rng(1).uniform(-1.0, 1.0, n)
    for (ap, aj, ax) in ((Ap, Aj, Ax), scaled(Ap, Aj, Ax, s)):
        A = sp.csr_matrix((ax, aj, ap), shape=(n, n))
        d = 1.0 / A.diagonal()
        for rtol in (1e-6, 1e-10):
            for dinv in (None, d):
                x, it, conv, brk = pcg_reference(ap, aj, ax, b, rtol, 4 * n, dinv)
                count = [0]
                xs, info = sla.cg(A, b, rtol=rtol, atol=0.0, maxiter=4 * n,
                                  M=None if dinv is None else sp.diags(dinv),
                                  callback=lambda xk: count.__setitem__(0, count[0] + 1))
                assert conv and not brk and info == 0
                assert it == count[0]
                np.testing.assert_allclose(x, xs, rtol=0, atol=1e-12 * np.abs(xs).max())


def test_reference_pcg_breakdown_and_edges():
    Ap, Aj, Ax = g.lap2d(8, np.float64)
    n = Ap.shape[0] - 1
    b = np.ones(n)
    x, it, conv, brk = pcg_reference(Ap, Aj, -Ax, b, 1e-8, n)
    assert (it, conv, brk) == (0, False, True) and np.all(x == 0)
    x, it, conv, brk = pcg_reference(Ap, Aj, Ax, np.zeros(n), 1e-8, n, x0=np.ones(n))
    assert (it, conv) == (0, True) and np.all(x == 0)
    x, it, conv, brk = pcg_reference(Ap, Aj, Ax, b, 1e-8, 0)
    assert (it, conv, brk) == (0, False, False)


def _valid_args(L_mod):
    a = L_mod.CgArgs()
    a.kind, a.offset_bits, a.value_bits, a.flags = 0, 32, 64, 0
    a.n, a.nnz = 4, 10
    a.Ap, a.Aj, a.Ax, a.b, a.x = 0x1000, 0x2000, 0x3000, 0x4000, 0x5000   # never dereferenced
    a.rtol, a.max_iter = 1e-6, 10
    return a


def test_cg_argument_validation_needs_no_device(built_lib):
    """Every invalid argument is refused with status 1 before any CUDA call."""
    from spmv_samples_b200 import _lib
    L = built_lib
    out = _lib.CgOut()

    def status(**changes):
        a = _valid_args(_lib)
        for k, v in changes.items():
            setattr(a, k, v)
        return L.spmvb200_cg(C.byref(a), C.byref(out))

    assert L.spmvb200_cg(None, C.byref(out)) == 1
    assert L.spmvb200_cg(C.byref(_valid_args(_lib)), None) == 1
    assert status(kind=6) == 1 and status(kind=-1) == 1             # unknown kind
    assert status(flags=2) == 1 and status(flags=3) == 1            # unknown flag bits
    for rtol in (0.0, -1e-6, float("nan")):
        assert status(rtol=rtol) == 1
    assert status(max_iter=-1) == 1
    for name in ("Ap", "Aj", "Ax", "b", "x"):
        assert status(**{name: None}) == 1, name                   # NULL with n > 0
    assert status(x=0x4000) == 1                                    # x == b
    assert status(n=-1) == 1 and status(nnz=-1) == 1
    assert status(Ap=0x1008) == 2                                   # the alignment rule of spmvb200_spmv
    assert status(value_bits=16) == 4
    # n == 0 is a no-op that converged in 0 iterations, pointers or not
    out.iterations, out.converged = 7, 0
    assert status(n=0, nnz=0, Ap=None, Aj=None, Ax=None, b=None, x=None) == 0
    assert out.iterations == 0 and out.converged == 1 and out.breakdown == 0


def test_solve_cg_checks_tensors_before_the_device():
    from spmv_samples_b200 import solve
    Ap, Aj, Ax = (torch.from_numpy(a) for a in g.lap2d(4, np.float64))
    b = torch.ones(16, dtype=torch.float64)
    with pytest.raises(TypeError):
        solve.cg(Ap, Aj, Ax, b.float())                          # b not of the matrix dtype
    with pytest.raises(TypeError):
        solve.cg(Ap, Aj.long(), Ax, b)                           # int64 column indices
    with pytest.raises(TypeError):
        solve.cg(Ap.short(), Aj, Ax, b)                          # int16 offsets
    with pytest.raises(TypeError):
        solve.cg(Ap, Aj, Ax, b, torch.zeros(16, dtype=torch.float32))
    with pytest.raises(ValueError, match="square"):
        Aj_wide = Aj.clone()
        Aj_wide[3] = 16                                          # a column beyond n: 16 x 17
        solve.cg(Ap, Aj_wide, Ax, b)
    with pytest.raises(ValueError, match="length"):
        solve.cg(Ap, Aj, Ax, torch.ones(15, dtype=torch.float64))
    with pytest.raises(ValueError, match="length"):
        solve.cg(Ap, Aj, Ax, b, torch.zeros(17, dtype=torch.float64))
    with pytest.raises(ValueError):
        solve.cg(Ap, Aj, Ax, b, rtol=0.0)
    with pytest.raises(ValueError):
        solve.cg(Ap, Aj, Ax, b, max_iter=-1)
    with pytest.raises(ValueError, match="CUDA"):
        solve.cg(Ap, Aj, Ax, b)                                  # well formed, but host tensors
