"""CPU suite for the restarted GMRES solve (spmvb200_gmres, spmv_samples_b200.solve.gmres): the
numpy restatement of the device algorithm that the GPU tests compare with, pinned to
scipy.sparse.linalg.gmres, and argument checks that need no device."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import cpu
from test_bicgstab_cpu import convdiff, jacobi_dinv, rmat_dominant, scaled_identity, swap_pairs
from test_cg_cpu import _valid_args


def gmres_reference(Ap, Aj, Ax, b, rtol, max_iter, restart, dinv=None, x0=None, eps=np.finfo(np.float64).eps,
                    trace=None):
    """Right-preconditioned GMRES(m) in fp64 on oracle.cpu.spmv_fp64, as csrc/gmres.cu runs it:
    m = min(restart, n); CGS2 (h = h1 + h2); rotations r = hypot(a, b), c = a / r, s = b / r
    (c = 1, s = 0 at r = 0); a cycle ends after m steps, at |g_{j+1}| <= rtol ||b||, at a lucky
    breakdown (||w|| after <= eps ||w|| before) or at the step cap, then x += M^-1 V y and the
    explicit ||b - A x|| decides.  Cycles are aligned to max_iter's step slots: one that ends
    early idles the rest of its m slots.  Breakdown: a non-finite h, norm or rotation (x stays at
    the cycle's start), a non-finite ||b|| or ||r0||, or a lucky breakdown whose explicit residual
    misses the tolerance.  trace, a list, gets one list of the |g_{j+1}| per cycle.  Returns
    (x, iterations, converged, breakdown)."""
    n = Ap.shape[0] - 1
    m = min(restart, n)
    b = np.asarray(b, dtype=np.float64)
    x = np.zeros(n) if x0 is None else np.array(x0, dtype=np.float64)

    def A(v):
        return cpu.spmv_fp64(Ap, Aj, Ax, v)

    def M(v):
        return v if dinv is None else dinv * v

    with np.errstate(all="ignore"):
        bnorm = np.linalg.norm(b)
        tol = rtol * bnorm
        r = b - A(x)
        beta = np.linalg.norm(r)
        if bnorm == 0:
            return np.zeros(n), 0, True, False
        if beta <= tol:
            return x, 0, True, False
        if not np.isfinite(bnorm) or not np.isfinite(beta):
            return x, 0, False, True
        it = slots = 0
        while slots < max_iter:
            cycle_slots = min(m, max_iter - slots)
            slots += cycle_slots
            V = np.zeros((m + 1, n))
            R = np.zeros((m, m))          # R[j, :j+1] = column j of the rotated Hessenberg matrix
            cs, sn = np.zeros(m), np.zeros(m)
            g = np.zeros(m + 1)
            g[0] = beta
            V[0] = r / beta
            k, lucky, est = 0, False, []
            for j in range(cycle_slots):
                w = A(M(V[j]))
                h1 = V[:j + 1] @ w
                h0 = np.linalg.norm(w)
                w = w - V[:j + 1].T @ h1
                h2 = V[:j + 1] @ w
                w = w - V[:j + 1].T @ h2
                hn = np.linalg.norm(w)
                col = h1 + h2
                finite = np.all(np.isfinite(col)) and np.isfinite(h0) and np.isfinite(hn)
                lucky = hn <= eps * h0
                if lucky:
                    hn = 0.0
                for i in range(j):
                    n0, n1 = col[i], col[i + 1]
                    col[i] = cs[i] * n0 + sn[i] * n1
                    col[i + 1] = -sn[i] * n0 + cs[i] * n1
                a = col[j]
                rr = np.hypot(a, hn)
                c, s = (1.0, 0.0) if rr == 0 else (a / rr, hn / rr)
                col[j] = rr
                gk1 = -s * g[j]
                if not (finite and np.all(np.isfinite(col)) and np.isfinite(c) and np.isfinite(s)
                        and np.isfinite(gk1)):
                    return x, it, False, True
                R[j, :j + 1] = col
                cs[j], sn[j] = c, s
                g[j], g[j + 1] = c * g[j], gk1
                est.append(abs(gk1))
                it += 1
                k = j + 1
                if lucky or abs(gk1) <= tol:
                    break
                V[j + 1] = w * (1.0 / hn)
            if trace is not None:
                trace.append(est)
            # y from R y = g, scipy's back substitution (a zero last pivot pseudo-solved)
            y = g[:k].copy()
            if R[k - 1, k - 1] == 0:
                y[k - 1] = 0.0
            for i in range(k - 1, 0, -1):
                if y[i] != 0:
                    y[i] /= R[i, i]
                    y[:i] -= y[i] * R[i, :i]
            if y[0] != 0:
                y[0] /= R[0, 0]
            x = x + M(y @ V[:k])
            r = b - A(x)
            beta = np.linalg.norm(r)
            if beta <= tol:
                return x, it, True, False
            if lucky or not np.isfinite(beta):
                return x, it, False, True
    return x, it, False, False


def scipy_gmres(Ap, Aj, Ax, b, rtol, restart):
    """scipy's solve (M = I) and its inner-iteration count (one pr_norm callback per step)."""
    sla = pytest.importorskip("scipy.sparse.linalg")
    sp = pytest.importorskip("scipy.sparse")
    n = Ap.shape[0] - 1
    A = sp.csr_matrix((Ax, Aj, Ap), shape=(n, n))
    seen = []
    xs, info = sla.gmres(A, b, rtol=rtol, atol=0.0, restart=restart, maxiter=10 * n,
                         callback=seen.append, callback_type="pr_norm")
    return xs, info, len(seen)


@pytest.mark.parametrize("restart", [64, 10])
@pytest.mark.parametrize("rtol", [1e-6, 1e-8])
@pytest.mark.parametrize("matrix", ["convdiff16", "rmat_dominant10"])
def test_reference_gmres_matches_scipy(matrix, rtol, restart):
    Ap, Aj, Ax = convdiff(16) if matrix == "convdiff16" else rmat_dominant(10)
    n = Ap.shape[0] - 1
    b = np.random.default_rng(1).uniform(-1.0, 1.0, n)
    x, it, conv, brk = gmres_reference(Ap, Aj, Ax, b, rtol, 10 * n, restart)
    xs, info, it_s = scipy_gmres(Ap, Aj, Ax, b, rtol, restart)
    assert conv and not brk and info == 0
    assert it == it_s, (it, it_s)
    np.testing.assert_allclose(x, xs, rtol=0, atol=1e-12 * np.abs(xs).max())


@pytest.mark.parametrize("restart", [64, 10, 3])
@pytest.mark.parametrize("matrix", ["convdiff16", "rmat_dominant10"])
def test_reference_gmres_estimates_never_increase_within_a_cycle(matrix, restart):
    Ap, Aj, Ax = convdiff(16) if matrix == "convdiff16" else rmat_dominant(10)
    n = Ap.shape[0] - 1
    b = np.random.default_rng(2).uniform(-1.0, 1.0, n)
    trace = []
    _, it, conv, _ = gmres_reference(Ap, Aj, Ax, b, 1e-8, 10 * n, restart, trace=trace)
    assert conv and sum(len(t) for t in trace) == it
    for est in trace:
        assert all(b_ <= a_ for a_, b_ in zip(est, est[1:])), est


def test_reference_gmres_lucky_breakdowns_and_edges():
    # swap pairs: the Krylov space of b is {even, odd}; converged in exactly 2 steps
    Ap, Aj, Ax = swap_pairs(8)
    b = np.where(np.arange(16) % 2 == 0, 1.0, 0.0)
    for restart in (64, 2):
        x, it, conv, brk = gmres_reference(Ap, Aj, Ax, b, 1e-14, 16, restart)
        assert (it, conv, brk) == (2, True, False)
        assert np.linalg.norm(b - cpu.spmv_fp64(Ap, Aj, Ax, x)) <= 1e-14 * np.linalg.norm(b)
    # restart 1 on swap pairs: each one-step cycle finds h = 0, stagnates, and runs out of steps
    x, it, conv, brk = gmres_reference(Ap, Aj, Ax, b, 1e-8, 5, 1)
    assert (it, conv, brk) == (5, False, False) and np.all(x == 0)
    # 4 I: one step, with and without Jacobi
    Ap, Aj, Ax = scaled_identity(16)
    b = np.random.default_rng(2).uniform(-1.0, 1.0, 16)
    for dinv in (None, jacobi_dinv(Ap, Aj, Ax)):
        x, it, conv, brk = gmres_reference(Ap, Aj, Ax, b, 1e-8, 16, 20, dinv)
        assert (it, conv, brk) == (1, True, False)
        np.testing.assert_allclose(x, b / 4, rtol=1e-15)
    # b = 0, x0 the solution, max_iter = 0
    Ap, Aj, Ax = convdiff(8)
    x, it, conv, _ = gmres_reference(Ap, Aj, Ax, np.zeros(64), 1e-8, 64, 20, x0=np.ones(64))
    assert (it, conv) == (0, True) and np.all(x == 0)
    x0 = np.arange(64, dtype=np.float64) % 5 - 2
    x, it, conv, _ = gmres_reference(Ap, Aj, Ax, cpu.spmv_fp64(Ap, Aj, Ax, x0), 1e-8, 64, 20, x0=x0)
    assert (it, conv) == (0, True) and np.array_equal(x, x0)
    x, it, conv, brk = gmres_reference(Ap, Aj, Ax, np.ones(64), 1e-8, 0, 20)
    assert (it, conv, brk) == (0, False, False)
    # NaN in b: breakdown before the first step
    bn = np.ones(64)
    bn[7] = np.nan
    x, it, conv, brk = gmres_reference(Ap, Aj, Ax, bn, 1e-8, 64, 20)
    assert (it, conv, brk) == (0, False, True)
    # a step cap inside a cycle: that many steps, x the minimiser over them
    full = gmres_reference(Ap, Aj, Ax, np.ones(64), 1e-10, 64, 20)
    assert full[2] and full[1] > 6
    short = gmres_reference(Ap, Aj, Ax, np.ones(64), 1e-10, full[1] - 3, 20)
    assert short[1:] == (full[1] - 3, False, False)


def test_reference_jacobi_needs_fewer_steps_on_rmat_dominant():
    Ap, Aj, Ax = rmat_dominant(10)
    n = Ap.shape[0] - 1
    b = np.random.default_rng(3).uniform(-1.0, 1.0, n)
    _, it_plain, conv_plain, _ = gmres_reference(Ap, Aj, Ax, b, 1e-10, n, 20)
    _, it_jac, conv_jac, _ = gmres_reference(Ap, Aj, Ax, b, 1e-10, n, 20, jacobi_dinv(Ap, Aj, Ax))
    assert conv_plain and conv_jac and it_jac < it_plain, (it_jac, it_plain)


def test_gmres_argument_validation_needs_no_device(built_lib):
    """The statuses of spmvb200_cg's validation, case for case, and the restart range, before any
    CUDA call."""
    from spmv_samples_b200 import _lib
    L = built_lib
    out = _lib.CgOut()

    def status(restart=20, **changes):
        a = _valid_args(_lib)
        for k, v in changes.items():
            setattr(a, k, v)
        return L.spmvb200_gmres(C.byref(a), restart, C.byref(out))

    assert L.spmvb200_gmres(None, 20, C.byref(out)) == 1
    assert L.spmvb200_gmres(C.byref(_valid_args(_lib)), 20, None) == 1
    for restart in (0, 65, -1):
        assert status(restart) == 1, restart
        assert status(restart, n=0, nnz=0, Ap=None, Aj=None, Ax=None, b=None, x=None) == 1, restart
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
    for restart in (1, 64):
        out.iterations, out.converged = 7, 0
        assert status(restart, n=0, nnz=0, Ap=None, Aj=None, Ax=None, b=None, x=None) == 0
        assert out.iterations == 0 and out.converged == 1 and out.breakdown == 0


def test_solve_gmres_checks_restart_and_tensors_before_the_device():
    from spmv_samples_b200 import solve
    Ap, Aj, Ax = (torch.from_numpy(a) for a in convdiff(4))
    b = torch.ones(16, dtype=torch.float64)
    for restart in (0, 65, -1, 2.0, True):
        with pytest.raises(ValueError, match="restart"):
            solve.gmres(Ap, Aj, Ax, b, restart=restart)
    with pytest.raises(TypeError):
        solve.gmres(Ap, Aj, Ax, b.float())
    with pytest.raises(ValueError, match="square"):
        Aj_wide = Aj.clone()
        Aj_wide[3] = 16
        solve.gmres(Ap, Aj_wide, Ax, b)
    with pytest.raises(ValueError, match="length"):
        solve.gmres(Ap, Aj, Ax, torch.ones(15, dtype=torch.float64))
    with pytest.raises(ValueError):
        solve.gmres(Ap, Aj, Ax, b, rtol=0.0)
    with pytest.raises(ValueError):
        solve.gmres(Ap, Aj, Ax, b, max_iter=-1)
    with pytest.raises(ValueError, match="different"):
        solve.gmres(Ap, Aj, Ax, b, b)
    with pytest.raises(ValueError, match="CUDA"):
        solve.gmres(Ap, Aj, Ax, b, restart=np.int64(30))
