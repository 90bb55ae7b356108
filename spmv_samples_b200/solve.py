"""Krylov solves of A x = b on the device: conjugate gradients (spmvb200_cg, csrc/cg.cu) for a
symmetric positive definite A; BiCGSTAB (spmvb200_bicgstab, csrc/bicgstab.cu) and restarted
GMRES (spmvb200_gmres, csrc/gmres.cu) for any square A.

    res = cg(Ap, Aj, Ax, b, rtol=1e-8, kind="auto", jacobi=True)
    res = bicgstab(Ap, Aj, Ax, b, rtol=1e-8, kind="auto", jacobi=True)
    res = gmres(Ap, Aj, Ax, b, rtol=1e-8, restart=30, kind="auto", jacobi=True)

A is an n x n CSR matrix (CUDA tensors, as for spmv.SpMV).  A CG iteration is one SpMV of the
chosen kind and three streaming kernels, a BiCGSTAB iteration two SpMVs and five, a GMRES step
one SpMV and four; the dot products accumulate in double in a fixed order, and the host reads the convergence flags once
per batch of iterations instead of once per iteration.  There is no PyTorch or CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import numbers
from dataclasses import dataclass

import torch

from . import _lib
from .spmv import _OFF, _VAL, KIND_IDS, SpMVKindError, _check_tensors


@dataclass
class CgResult:
    x: torch.Tensor        # the solution (the caller's x, updated in place, when one was given)
    iterations: int
    residual_norm: float   # ||b - A x|| of the returned x, computed in fp64
    b_norm: float
    converged: bool        # ||r|| <= rtol * ||b||: the recursive r (cg, bicgstab), the explicit one (gmres)
    breakdown: bool        # the method cannot continue (not an error): see each solver


def cg(Ap, Aj, Ax, b, x=None, *, rtol=1e-6, max_iter=None, kind="auto", jacobi=False,
       stream=None) -> CgResult:
    """Solve A x = b by conjugate gradients, Jacobi-preconditioned (M = diag(A)) with jacobi=True.
    x: initial guess, overwritten with the solution; None starts from zero.  max_iter: None means
    n.  Stops at the first iteration with ||r|| <= rtol * ||b||, after max_iter iterations, or at a
    breakdown.  Raises SpmvB200Error (status 1) when jacobi=True and a diagonal entry is missing or
    zero."""
    return _solve("spmvb200_cg", Ap, Aj, Ax, b, x, rtol, max_iter, kind, jacobi, stream)


def bicgstab(Ap, Aj, Ax, b, x=None, *, rtol=1e-6, max_iter=None, kind="auto", jacobi=False,
             stream=None) -> CgResult:
    """Solve A x = b for a general square A by right-preconditioned BiCGSTAB, with M = diag(A)
    when jacobi=True, in the operation order of scipy.sparse.linalg.bicgstab.  x: initial guess,
    overwritten with the solution; None starts from zero.  max_iter: None means n.  Stops when
    ||r|| <= rtol * ||b|| (also at the half step, ||s|| <= rtol * ||b||, which counts as an
    iteration), after max_iter iterations, or at a breakdown: an exact zero or a non-finite value
    of one of the method's scalars, which leaves x at its last finite iterate.  Raises
    SpmvB200Error (status 1) when jacobi=True and a diagonal entry is missing or zero."""
    return _solve("spmvb200_bicgstab", Ap, Aj, Ax, b, x, rtol, max_iter, kind, jacobi, stream)


def gmres(Ap, Aj, Ax, b, x=None, *, rtol=1e-6, restart=20, max_iter=None, kind="auto", jacobi=False,
          stream=None) -> CgResult:
    """Solve A x = b for a general square A by right-preconditioned restarted GMRES(restart), with
    M = diag(A) when jacobi=True.  Right preconditioning minimises the true residual, so rtol
    means what it means for cg() (scipy.sparse.linalg.gmres preconditions on the left).  Each
    cycle orthogonalises by classical Gram-Schmidt with one re-orthogonalisation and ends after
    min(restart, n) steps, when the residual estimate meets rtol * ||b||, or at a lucky breakdown;
    then the explicit ||b - A x|| decides convergence or starts the next cycle.  restart: 1 to 64.
    x: initial guess, overwritten with the solution; None starts from zero.  max_iter: the cap on
    Arnoldi steps, which `iterations` counts (the idle rest of a cycle that ended early counts
    against it); None means n.  A breakdown is a non-finite value in the method (x is left at the
    start of that cycle) or a lucky breakdown whose explicit residual misses the tolerance.
    Raises ValueError for a restart outside [1, 64], and SpmvB200Error (status 1) when
    jacobi=True and a diagonal entry is missing or zero."""
    if isinstance(restart, bool) or not isinstance(restart, numbers.Integral) or not 1 <= restart <= _lib.GMRES_MAX_RESTART:
        raise ValueError(f"restart must be an integer in [1, {_lib.GMRES_MAX_RESTART}]")
    return _solve("spmvb200_gmres", Ap, Aj, Ax, b, x, rtol, max_iter, kind, jacobi, stream, int(restart))


def _solve(entry, Ap, Aj, Ax, b, x, rtol, max_iter, kind, jacobi, stream, *extra) -> CgResult:
    """Every solver: the argument checks, made before touching a device, then the call, with the
    solver's own arguments (`extra`) between the records."""
    for name, t in (("Ap", Ap), ("Aj", Aj), ("Ax", Ax), ("b", b), ("x", x)):
        if t is not None and t.dim() != 1:
            raise ValueError(f"{name} must be 1-D")
    if Ap.dtype not in _OFF:
        raise TypeError(f"offset type {Ap.dtype} unsupported (int32 / int64)")
    if Aj.dtype != torch.int32:
        raise TypeError("index type must be int32")
    if Ax.dtype not in _VAL or b.dtype != Ax.dtype or (x is not None and x.dtype != Ax.dtype):
        raise TypeError("Ax, b, x must share one dtype, float32 or float64")
    n = Ap.numel() - 1
    if n < 0:
        raise ValueError("Ap must hold n + 1 offsets")
    if Ax.numel() != Aj.numel():
        raise ValueError("Aj and Ax must have the same length")
    if b.numel() != n or (x is not None and x.numel() != n):
        raise ValueError(f"b and x must have length n = {n}")
    if Aj.numel() and (int(Aj.min()) < 0 or int(Aj.max()) >= n):
        raise ValueError(f"A must be square: column indices must lie in [0, {n})")
    if kind not in KIND_IDS:
        raise SpMVKindError(f'SpMV kind "{kind}" is NOT SUPPROT')
    if not rtol > 0:
        raise ValueError("rtol must be positive")
    if max_iter is None:
        max_iter = n
    if max_iter < 0:
        raise ValueError("max_iter must be >= 0")
    if x is None:
        x = torch.zeros_like(b)
    elif x.data_ptr() == b.data_ptr() and n > 0:
        raise ValueError("x and b must be different tensors")
    _check_tensors(Ap, Aj, Ax, b, x)

    a = _lib.CgArgs()
    a.kind = KIND_IDS[kind]
    a.offset_bits = _OFF[Ap.dtype][1]
    a.value_bits = _VAL[Ax.dtype][1]
    a.flags = _lib.CG_JACOBI if jacobi else 0
    a.n, a.nnz = n, Aj.numel()
    a.Ap, a.Aj, a.Ax, a.b, a.x = Ap.data_ptr(), Aj.data_ptr(), Ax.data_ptr(), b.data_ptr(), x.data_ptr()
    a.rtol = float(rtol)
    a.max_iter = int(max_iter)
    a.stream = (stream if stream is not None else torch.cuda.current_stream(Ap.device)).cuda_stream
    out = _lib.CgOut()
    with torch.cuda.device(Ap.device):
        st = getattr(_lib.lib(), entry)(C.byref(a), *extra, C.byref(out))
    _lib.check(st, f"{entry}[{kind}]")
    return CgResult(x=x, iterations=int(out.iterations), residual_norm=float(out.residual_norm),
                    b_norm=float(out.b_norm), converged=bool(out.converged), breakdown=bool(out.breakdown))
