"""GPU suite for the conjugate-gradient solve (spmvb200_cg through spmv_samples_b200.solve.cg):
accuracy against the fp64 numpy restatement of PCG (tests/test_cg_cpu.py), determinism, exact
early exit, edge cases, breakdown, the Jacobi diagonal check, the launch count, and bin/spmv --cg."""
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import cpu
from oracle import generators as g
from test_cg_cpu import pcg_reference, scaled

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "bin", "spmv")
MAX_BATCH = 64   # kCgMaxBatch in csrc/cg.cu: iterations enqueued between two reads of the flags


@pytest.fixture(scope="module", autouse=True)
def _device(built_lib):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    torch.cuda.set_device(0)
    yield
    from spmv_samples_b200 import spmv
    spmv.release_cache()


_cache = {}


def problem(grid, dtype=np.float64, offset=np.int32, s=None):
    """lap2d(grid) (or S A S), and b = A x_true for a seeded x_true in [-1, 1]: host arrays in
    the value type, plus their device copies."""
    key = (grid, np.dtype(dtype).name, np.dtype(offset).name, s is not None)
    if key not in _cache:
        Ap, Aj, Ax = g.lap2d(grid, np.float64, offset)
        if s is not None:
            Ap, Aj, Ax = scaled(Ap, Aj, Ax, s)
        Ax = Ax.astype(dtype)
        n = Ap.shape[0] - 1
        x_true = np.random.default_rng(grid).uniform(-1.0, 1.0, n)
        b = cpu.spmv_fp64(Ap, Aj, Ax, x_true).astype(dtype)
        dev = tuple(torch.from_numpy(a).cuda() for a in (Ap, Aj, Ax, b))
        _cache[key] = (Ap, Aj, Ax, b, dev)
    return _cache[key]


def true_residual(Ap, Aj, Ax, b, x):
    return float(np.linalg.norm(b.astype(np.float64) - cpu.spmv_fp64(Ap, Aj, Ax, x.cpu().numpy())))


@pytest.mark.parametrize("kind", ["merge", "vector", "light", "stream", "auto"])
@pytest.mark.parametrize("offset", [np.int32, np.int64], ids=["o32", "o64"])
@pytest.mark.parametrize("grid", [64, 128])
def test_cg_f64_accuracy(grid, offset, kind):
    from spmv_samples_b200 import solve
    rtol = 1e-8
    Ap, Aj, Ax, b, dev = problem(grid, np.float64, offset)
    res = solve.cg(*dev, rtol=rtol, kind=kind)
    _, it_ref, conv_ref, _ = pcg_reference(Ap, Aj, Ax, b, rtol, Ap.shape[0] - 1)
    assert res.converged and not res.breakdown and conv_ref
    assert abs(res.iterations - it_ref) <= 2, (res.iterations, it_ref)
    bn = float(np.linalg.norm(b))
    assert res.b_norm == pytest.approx(bn, rel=1e-12)
    tr = true_residual(Ap, Aj, Ax, b, res.x)
    assert tr <= 1.01 * rtol * bn, (tr, rtol * bn)
    assert res.residual_norm == pytest.approx(tr, rel=1e-10)


@pytest.mark.parametrize("kind", ["merge", "auto"])
def test_cg_f32(kind):
    from spmv_samples_b200 import solve
    rtol = 1e-4
    Ap, Aj, Ax, b, dev = problem(128, np.float32)
    res = solve.cg(*dev, rtol=rtol, kind=kind)
    assert res.converged and not res.breakdown
    tr = true_residual(Ap, Aj, Ax, b, res.x)
    assert tr <= 2 * rtol * float(np.linalg.norm(b.astype(np.float64)))
    assert res.residual_norm == pytest.approx(tr, rel=1e-10)   # fp64 on both sides, from the same x


def test_cg_jacobi_on_a_badly_scaled_matrix():
    from spmv_samples_b200 import solve
    rtol = 1e-8
    s = np.random.default_rng(7).uniform(1.0, 10.0, 64 * 64)
    Ap, Aj, Ax, b, dev = problem(64, np.float64, np.int32, s)
    plain = solve.cg(*dev, rtol=rtol, kind="auto")
    jac = solve.cg(*dev, rtol=rtol, kind="auto", jacobi=True)
    assert plain.converged and jac.converged
    assert jac.iterations < plain.iterations, (jac.iterations, plain.iterations)
    rows = np.repeat(np.arange(Ap.shape[0] - 1), np.diff(Ap))
    dinv = 1.0 / Ax[Aj == rows]
    _, it_ref, _, _ = pcg_reference(Ap, Aj, Ax, b, rtol, Ap.shape[0] - 1, dinv)
    assert abs(jac.iterations - it_ref) <= 2, (jac.iterations, it_ref)
    assert true_residual(Ap, Aj, Ax, b, jac.x) <= 1.01 * rtol * float(np.linalg.norm(b))


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("kind", ["merge", "vector", "auto"])
def test_cg_is_deterministic(kind, dtype):
    from spmv_samples_b200 import solve
    _, _, _, _, dev = problem(64, dtype)
    rtol = 1e-4 if dtype == np.float32 else 1e-8
    a = solve.cg(*dev, rtol=rtol, kind=kind, jacobi=True)
    b = solve.cg(*dev, rtol=rtol, kind=kind, jacobi=True)
    assert a.iterations == b.iterations and a.residual_norm == b.residual_norm
    assert torch.equal(a.x, b.x)


def test_cg_early_exit_is_exact():
    """The flags stop every CG kernel of an iteration batch already enqueued: the solve that
    stops at m returns the same bits as one allowed exactly m iterations."""
    from spmv_samples_b200 import solve
    _, _, _, _, dev = problem(64)
    n = dev[0].numel() - 1
    full = solve.cg(*dev, rtol=1e-8, kind="auto", max_iter=n)
    m = full.iterations
    assert full.converged and m > 10
    exact = solve.cg(*dev, rtol=1e-8, kind="auto", max_iter=m)
    assert exact.converged and exact.iterations == m and torch.equal(exact.x, full.x)
    short = solve.cg(*dev, rtol=1e-8, kind="auto", max_iter=m - 3)
    assert short.iterations == m - 3 and not short.converged and not short.breakdown


def test_cg_edge_cases():
    from spmv_samples_b200 import solve
    Ap, Aj, Ax, b, dev = problem(32)
    dAp, dAj, dAx, db = dev
    n = Ap.shape[0] - 1
    # b = 0: x = 0 whatever x0 was
    res = solve.cg(dAp, dAj, dAx, torch.zeros_like(db), torch.ones_like(db), rtol=1e-8)
    assert res.converged and res.iterations == 0 and res.b_norm == 0.0
    assert torch.count_nonzero(res.x) == 0
    # x0 already the solution (integer x: A x0 is exact)
    x0 = np.random.default_rng(5).integers(-3, 4, n).astype(np.float64)
    bx = torch.from_numpy(cpu.spmv_fp64(Ap, Aj, Ax, x0)).cuda()
    x = torch.from_numpy(x0).cuda()
    res = solve.cg(dAp, dAj, dAx, bx, x, rtol=1e-8)
    assert res.converged and res.iterations == 0 and res.residual_norm == 0.0
    assert res.x is x and torch.equal(x.cpu(), torch.from_numpy(x0))
    # n = 0
    e = torch.zeros(0, dtype=torch.float64, device="cuda")
    res = solve.cg(torch.zeros(1, dtype=torch.int32, device="cuda"),
                   torch.zeros(0, dtype=torch.int32, device="cuda"), e, e.clone())
    assert res.converged and res.iterations == 0 and res.x.numel() == 0
    # max_iter = 0: nothing moves, the residual is that of x0 = 0
    res = solve.cg(*dev, rtol=1e-8, max_iter=0)
    assert not res.converged and not res.breakdown and res.iterations == 0
    assert torch.count_nonzero(res.x) == 0
    assert res.residual_norm == pytest.approx(float(np.linalg.norm(b)), rel=1e-12)


@pytest.mark.parametrize("jacobi", [False, True])
def test_cg_breakdown_on_negative_definite(jacobi):
    from spmv_samples_b200 import solve
    _, _, _, _, (dAp, dAj, dAx, db) = problem(32)
    res = solve.cg(dAp, dAj, -dAx, db, rtol=1e-8, jacobi=jacobi)
    assert res.breakdown and not res.converged
    assert bool(torch.isfinite(res.x).all())


@pytest.mark.parametrize("jacobi", [False, True])
@pytest.mark.parametrize("poison", ["nan_in_b", "inf_in_x0", "nan_off_diagonal"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
def test_cg_non_finite_input_breaks_down_at_once(dtype, poison, jacobi):
    """A NaN or an inf present from the start makes r.z (or ||b||) non-finite in the set-up: the
    solve reports a breakdown before the first iteration instead of iterating on NaN."""
    from spmv_samples_b200 import solve
    Ap, Aj, Ax, b, (dAp, dAj, dAx, db) = problem(32, dtype)
    n = Ap.shape[0] - 1
    x0 = torch.zeros_like(db)
    if poison == "nan_in_b":
        db = db.clone()
        db[n // 2] = float("nan")
    elif poison == "inf_in_x0":
        x0[n // 3] = float("inf")
    else:
        rows = np.repeat(np.arange(n), np.diff(Ap))
        k = int(np.nonzero(Aj != rows)[0][len(Aj) // 3])
        dAx = dAx.clone()
        dAx[k] = float("nan")
    res = solve.cg(dAp, dAj, dAx, db, x0, rtol=1e-6, jacobi=jacobi)
    assert res.breakdown and not res.converged and res.iterations == 0, res


def test_cg_jacobi_rejects_a_bad_diagonal():
    from spmv_samples_b200 import _lib, solve
    Ap, Aj, Ax, b, _ = problem(16)
    rows = np.repeat(np.arange(Ap.shape[0] - 1), np.diff(Ap))
    diag = np.nonzero(Aj == rows)[0]
    zero = Ax.copy()
    zero[diag[5]] = 0.0                                              # A[5,5] = 0
    keep = np.ones(Aj.shape[0], bool)
    keep[diag[9]] = False                                            # A[9,9] missing
    Ap_m = np.concatenate([[0], np.cumsum(np.bincount(rows[keep], minlength=Ap.shape[0] - 1))]).astype(Ap.dtype)
    for ap, aj, ax in ((Ap, Aj, zero), (Ap_m, Aj[keep], Ax[keep])):
        d = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (ap, aj, ax, b)]
        with pytest.raises(_lib.SpmvB200Error) as e:
            solve.cg(*d, rtol=1e-8, jacobi=True)
        assert e.value.status == 1
        assert solve.cg(*d, rtol=1e-8, max_iter=3).iterations <= 3   # without Jacobi it runs


@pytest.mark.parametrize("kind", ["merge", "vector", "auto"])
def test_cg_launch_count(kind):
    """One SpMV and three kernels per iteration; past the last one, at most one batch of
    iterations whose kernels return at once, plus the set-up and the final residual."""
    from spmv_samples_b200 import solve, spmv
    _, _, _, _, dev = problem(64)
    dAp, dAj, dAx, db = dev
    y = torch.empty_like(db)
    spmv.spmv_ex(kind, dAp, dAj, dAx, db, y)
    spmv.spmv_ex(kind, dAp, dAj, dAx, db, y, static_pattern=True)
    before = spmv.launch_count()
    spmv.spmv_ex(kind, dAp, dAj, dAx, db, y, static_pattern=True)
    per_spmv = spmv.launch_count() - before
    solve.cg(*dev, rtol=1e-8, kind=kind)   # warm: statistics cache, scratch
    before = spmv.launch_count()
    res = solve.cg(*dev, rtol=1e-8, kind=kind)
    launched = spmv.launch_count() - before
    assert res.converged
    assert launched >= res.iterations * (per_spmv + 3)
    assert launched <= (res.iterations + MAX_BATCH) * (per_spmv + 3) + 8, (launched, res.iterations, per_spmv)


def test_driver_cg():
    if not os.path.exists(BIN):
        subprocess.run(["make", "-C", ROOT, "-s", "bin/spmv"], check=True)
    r = subprocess.run([BIN, "synthetic:c1:256", "auto", "merge", "--iters", "20", "--cg", "1e-6"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = [ln for ln in r.stdout.splitlines() if "iterations" in ln and "CONVERGED" in ln]
    assert len(lines) == 2, r.stdout
    its = [int(ln.split("]")[1].split()[0]) for ln in lines]
    assert all(i > 0 for i in its)
    r = subprocess.run([BIN, "synthetic:c1", "auto", "--iters", "20", "--cg", "1e-6", "--jacobi"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Jacobi" in r.stdout and "CONVERGED" in r.stdout
