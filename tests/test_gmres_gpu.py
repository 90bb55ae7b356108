"""GPU suite for the restarted GMRES solve (spmvb200_gmres through spmv_samples_b200.solve.gmres):
accuracy against the fp64 numpy restatement (tests/test_gmres_cpu.py), fp32, Jacobi, the lucky
breakdown where BiCGSTAB breaks down, restarts, exact early exit, determinism, the table plan of
the merge kernel, edge cases, non-finite input, the Jacobi diagonal check, the launch count, and
bin/spmv --gmres."""
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import cpu
from test_bicgstab_cpu import convdiff, jacobi_dinv, rmat_dominant, scaled_identity, swap_pairs
from test_bicgstab_gpu import _write_mtx, problem, true_residual
from test_gmres_cpu import gmres_reference

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "bin", "spmv")
MAX_BATCH = 64   # kKrylovMaxBatch in csrc/krylov.cuh: step slots enqueued between two reads of the flags


@pytest.fixture(scope="module", autouse=True)
def _device(built_lib):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    torch.cuda.set_device(0)
    yield
    from spmv_samples_b200 import spmv
    spmv.release_cache()


@pytest.mark.parametrize("kind", ["merge", "vector", "light", "stream", "auto"])
@pytest.mark.parametrize("offset", [np.int32, np.int64], ids=["o32", "o64"])
@pytest.mark.parametrize("grid", [64, 128])
def test_gmres_f64_accuracy(grid, offset, kind):
    from spmv_samples_b200 import solve
    rtol = 1e-8
    Ap, Aj, Ax, b, dev = problem(f"convdiff{grid}", np.float64, offset)
    res = solve.gmres(*dev, rtol=rtol, restart=20, kind=kind)
    _, it_ref, conv_ref, _ = gmres_reference(Ap, Aj, Ax, b, rtol, Ap.shape[0] - 1, 20)
    assert res.converged and not res.breakdown and conv_ref
    assert abs(res.iterations - it_ref) <= 2, (res.iterations, it_ref)
    bn = float(np.linalg.norm(b))
    assert res.b_norm == pytest.approx(bn, rel=1e-12)
    tr = true_residual(Ap, Aj, Ax, b, res.x)
    assert tr <= 1.01 * rtol * bn, (tr, rtol * bn)
    assert res.residual_norm == pytest.approx(tr, rel=1e-10)


@pytest.mark.parametrize("kind", ["merge", "auto"])
def test_gmres_f32(kind):
    from spmv_samples_b200 import solve
    rtol = 1e-4
    Ap, Aj, Ax, b, dev = problem("convdiff128", np.float32)
    res = solve.gmres(*dev, rtol=rtol, restart=30, kind=kind)
    assert res.converged and not res.breakdown
    tr = true_residual(Ap, Aj, Ax, b, res.x)
    assert tr <= 2 * rtol * float(np.linalg.norm(b.astype(np.float64)))
    assert res.residual_norm == pytest.approx(tr, rel=1e-10)


def test_gmres_jacobi_on_rmat_dominant():
    from spmv_samples_b200 import solve
    rtol = 1e-10
    Ap, Aj, Ax, b, dev = problem("rmat14")
    plain = solve.gmres(*dev, rtol=rtol, kind="auto")
    jac = solve.gmres(*dev, rtol=rtol, kind="auto", jacobi=True)
    assert plain.converged and jac.converged
    assert jac.iterations < plain.iterations, (jac.iterations, plain.iterations)
    _, it_ref, _, _ = gmres_reference(Ap, Aj, Ax, b, rtol, Ap.shape[0] - 1, 20, jacobi_dinv(Ap, Aj, Ax))
    assert abs(jac.iterations - it_ref) <= 2, (jac.iterations, it_ref)
    assert true_residual(Ap, Aj, Ax, b, jac.x) <= 1.01 * rtol * float(np.linalg.norm(b))


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
def test_gmres_solves_swap_pairs_where_bicgstab_breaks_down(dtype):
    """The Krylov space of b is {even, odd}: the second step is a lucky breakdown, and x is the
    exact solution."""
    from spmv_samples_b200 import solve
    Ap, Aj, Ax = swap_pairs(1000, dtype)
    b = np.where(np.arange(2000) % 2 == 0, 1.0, 0.0).astype(dtype)
    dev = [torch.from_numpy(a).cuda() for a in (Ap, Aj, Ax, b)]
    assert solve.bicgstab(*dev, rtol=1e-8).breakdown
    bound = 1e-6 if dtype == np.float32 else 1e-14
    res = solve.gmres(*dev, rtol=bound)
    assert res.converged and not res.breakdown and res.iterations == 2, res
    assert true_residual(Ap, Aj, Ax, b, res.x) <= bound * float(np.linalg.norm(b))


@pytest.mark.parametrize("jacobi", [False, True])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
def test_gmres_one_step_on_4_identity(dtype, jacobi):
    from spmv_samples_b200 import solve
    Ap, Aj, Ax = scaled_identity(5000, 4.0, dtype)
    b = np.random.default_rng(4).uniform(-1.0, 1.0, 5000).astype(dtype)
    res = solve.gmres(*[torch.from_numpy(a).cuda() for a in (Ap, Aj, Ax, b)], rtol=1e-6, jacobi=jacobi)
    assert res.converged and not res.breakdown and res.iterations == 1, res
    np.testing.assert_allclose(res.x.cpu().numpy(), b / dtype(4), rtol=1e-5 if dtype == np.float32 else 1e-13)


def test_gmres_restarts_never_increase_the_residual():
    """GMRES(10) stopped after 10, 20, ... 50 steps: each cycle minimises the residual over a space
    that holds the previous iterate, so the explicit residual does not grow."""
    from spmv_samples_b200 import solve
    _, _, _, _, dev = problem("convdiff64")
    norms = []
    for cycles in range(1, 6):
        res = solve.gmres(*dev, rtol=1e-14, restart=10, max_iter=10 * cycles, kind="auto")
        assert res.iterations == 10 * cycles and not res.converged and not res.breakdown
        norms.append(res.residual_norm)
    assert all(b_ <= a_ * (1 + 1e-12) for a_, b_ in zip(norms, norms[1:])), norms
    assert norms[-1] < norms[0]


def test_gmres_early_exit_is_exact():
    """A cycle that converges early idles to its end on the device: the solve that stops at m
    returns the same bits as one allowed exactly m steps."""
    from spmv_samples_b200 import solve
    _, _, _, _, dev = problem("convdiff64")
    full = solve.gmres(*dev, rtol=1e-8, restart=20, kind="auto")
    m = full.iterations
    assert full.converged and m > 40
    exact = solve.gmres(*dev, rtol=1e-8, restart=20, kind="auto", max_iter=m)
    assert exact.converged and exact.iterations == m and torch.equal(exact.x, full.x)
    short = solve.gmres(*dev, rtol=1e-8, restart=20, kind="auto", max_iter=m - 3)
    assert short.iterations == m - 3 and not short.converged and not short.breakdown


@pytest.mark.parametrize("jacobi", [False, True])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("kind", ["merge", "vector", "auto"])
def test_gmres_is_deterministic(kind, dtype, jacobi):
    from spmv_samples_b200 import solve
    _, _, _, _, dev = problem("convdiff64", dtype)
    rtol = 1e-4 if dtype == np.float32 else 1e-8
    a = solve.gmres(*dev, rtol=rtol, kind=kind, jacobi=jacobi)
    b = solve.gmres(*dev, rtol=rtol, kind=kind, jacobi=jacobi)
    assert a.converged
    assert a.iterations == b.iterations and a.residual_norm == b.residual_norm
    assert torch.equal(a.x, b.x)


def test_gmres_on_the_table_plan():
    """R-MAT scale 20 in fp32 with kind merge: the static-pattern SpMVs build the table plan
    (csrc/hotx.cu) and the persistent table kernel runs the SpMV of every step, on a new basis
    vector each time.  150 steps (short of convergence at rtol 1e-4) are bit-identical to the ones
    with the table off."""
    from spmv_samples_b200 import solve, spmv
    Ap, Aj, Ax = rmat_dominant(20, 16, 3, np.float32)
    n = Ap.shape[0] - 1
    b = cpu.spmv_fp64(Ap, Aj, Ax, np.random.default_rng(20).uniform(-1.0, 1.0, n)).astype(np.float32)
    dev = [torch.from_numpy(a).cuda() for a in (Ap, Aj, Ax, b)]
    rtol = 1e-4
    spmv.release_cache()
    with_table = solve.gmres(*dev, rtol=rtol, restart=30, max_iter=150, kind="merge")
    info = spmv.hot_x_info(dev[1])
    assert info["table_columns"] > 0, info
    old = spmv.get_option("hot_x_table")
    spmv.set_option("hot_x_table", 0)
    try:
        spmv.release_cache()
        plain = solve.gmres(*dev, rtol=rtol, restart=30, max_iter=150, kind="merge")
        assert spmv.hot_x_info(dev[1])["table_columns"] == 0
    finally:
        spmv.set_option("hot_x_table", old)
        spmv.release_cache()
    assert with_table.iterations == plain.iterations == 150 and not with_table.breakdown
    assert with_table.residual_norm == plain.residual_norm
    assert torch.equal(with_table.x, plain.x)


def test_gmres_edge_cases():
    from spmv_samples_b200 import solve
    Ap, Aj, Ax, b, dev = problem("convdiff32")
    dAp, dAj, dAx, db = dev
    n = Ap.shape[0] - 1
    # b = 0: x = 0 whatever x0 was
    res = solve.gmres(dAp, dAj, dAx, torch.zeros_like(db), torch.ones_like(db), rtol=1e-8)
    assert res.converged and res.iterations == 0 and res.b_norm == 0.0
    assert torch.count_nonzero(res.x) == 0
    # x0 already the solution (integer x: A x0 is exact)
    x0 = np.random.default_rng(5).integers(-3, 4, n).astype(np.float64)
    bx = torch.from_numpy(cpu.spmv_fp64(Ap, Aj, Ax, x0)).cuda()
    x = torch.from_numpy(x0).cuda()
    res = solve.gmres(dAp, dAj, dAx, bx, x, rtol=1e-8)
    assert res.converged and res.iterations == 0 and res.residual_norm == 0.0
    assert res.x is x and torch.equal(x.cpu(), torch.from_numpy(x0))
    # n = 0
    e = torch.zeros(0, dtype=torch.float64, device="cuda")
    res = solve.gmres(torch.zeros(1, dtype=torch.int32, device="cuda"),
                      torch.zeros(0, dtype=torch.int32, device="cuda"), e, e.clone())
    assert res.converged and res.iterations == 0 and res.x.numel() == 0
    # max_iter = 0: nothing moves, the residual is that of x0 = 0
    res = solve.gmres(*dev, rtol=1e-8, max_iter=0)
    assert not res.converged and not res.breakdown and res.iterations == 0
    assert torch.count_nonzero(res.x) == 0
    assert res.residual_norm == pytest.approx(float(np.linalg.norm(b)), rel=1e-12)
    # restart above n: cycles of n steps
    Ap2, Aj2, Ax2 = convdiff(4)
    b2 = np.random.default_rng(6).uniform(-1.0, 1.0, 16)
    res = solve.gmres(*[torch.from_numpy(a).cuda() for a in (Ap2, Aj2, Ax2, b2)], rtol=1e-12, restart=64)
    _, it_ref, _, _ = gmres_reference(Ap2, Aj2, Ax2, b2, 1e-12, 16, 64)
    assert res.converged and abs(res.iterations - it_ref) <= 1 and res.iterations <= 16


@pytest.mark.parametrize("jacobi", [False, True])
@pytest.mark.parametrize("poison", ["nan_in_b", "inf_in_x0", "nan_off_diagonal"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
def test_gmres_non_finite_input_breaks_down_at_once(dtype, poison, jacobi):
    """A NaN or an inf present from the start makes ||b|| or ||r0|| non-finite in the set-up:
    the solve reports a breakdown before the first step."""
    from spmv_samples_b200 import solve
    Ap, Aj, Ax, b, (dAp, dAj, dAx, db) = problem("convdiff32", dtype)
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
    res = solve.gmres(dAp, dAj, dAx, db, x0, rtol=1e-6, jacobi=jacobi)
    assert res.breakdown and not res.converged and res.iterations == 0, res


def test_gmres_jacobi_rejects_a_bad_diagonal():
    from spmv_samples_b200 import _lib, solve
    Ap, Aj, Ax, b, _ = problem("convdiff16")
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
            solve.gmres(*d, rtol=1e-8, jacobi=True)
        assert e.value.status == 1
        assert solve.gmres(*d, rtol=1e-8, max_iter=3).iterations <= 3   # without Jacobi it runs


def _static_spmv_launches(kind, dev):
    from spmv_samples_b200 import spmv
    dAp, dAj, dAx, db = dev
    y = torch.empty_like(db)
    spmv.spmv_ex(kind, dAp, dAj, dAx, db, y)
    spmv.spmv_ex(kind, dAp, dAj, dAx, db, y, static_pattern=True)
    before = spmv.launch_count()
    spmv.spmv_ex(kind, dAp, dAj, dAx, db, y, static_pattern=True)
    return spmv.launch_count() - before


@pytest.mark.parametrize("kind", ["merge", "vector", "auto"])
def test_gmres_launches_per_step_do_not_grow_with_the_basis(kind):
    """Within one cycle, every Arnoldi step is one SpMV and four kernels, whether the basis holds
    2 vectors or 40: the launches of a 40-step cycle exceed those of a 4-step one by exactly
    36 steps' worth."""
    from spmv_samples_b200 import solve, spmv
    _, _, _, _, dev = problem("convdiff64")
    per_spmv = _static_spmv_launches(kind, dev)
    solve.gmres(*dev, rtol=1e-14, restart=64, max_iter=4, kind=kind)   # warm: statistics cache, scratch
    counts = {}
    for steps in (4, 40):
        before = spmv.launch_count()
        res = solve.gmres(*dev, rtol=1e-14, restart=64, max_iter=steps, kind=kind)
        counts[steps] = spmv.launch_count() - before
        assert res.iterations == steps and not res.converged
    assert counts[40] - counts[4] == 36 * (per_spmv + 4), (counts, per_spmv)


@pytest.mark.parametrize("kind", ["merge", "vector", "auto"])
def test_gmres_launch_count(kind):
    """The bound in csrc/gmres.cu: the set-up, one SpMV + 4 kernels per enqueued step slot, one
    SpMV + 3 kernels per cycle end, the final residual; the slots run past the converging
    step by at most the rest of its cycle and one batch."""
    from spmv_samples_b200 import solve, spmv
    _, _, _, _, dev = problem("convdiff64")
    n = dev[0].numel() - 1
    per_spmv = _static_spmv_launches(kind, dev)
    m = 20
    solve.gmres(*dev, rtol=1e-8, restart=m, kind=kind)   # warm
    before = spmv.launch_count()
    res = solve.gmres(*dev, rtol=1e-8, restart=m, kind=kind)
    launched = spmv.launch_count() - before
    assert res.converged
    it = res.iterations
    assert launched >= it * (per_spmv + 4) + -(-it // m) * (per_spmv + 3)
    slots = min(n, -(-it // m) * m + MAX_BATCH)
    bound = (per_spmv + 2 + 8) + slots * (per_spmv + 4) + -(-slots // m) * (per_spmv + 3) + 1
    assert launched <= bound, (launched, bound, it, per_spmv)


def test_driver_gmres(tmp_path):
    """c1 is an fp32 Laplacian with b = A*1: its fp32 explicit residual b - A x stalls near
    1e-6 * ||b|| (the rounding of the fp32 SpMV), and GMRES judges convergence by that residual,
    so the solve asks for 1e-5."""
    if not os.path.exists(BIN):
        subprocess.run(["make", "-C", ROOT, "-s", "bin/spmv"], check=True)
    r = subprocess.run([BIN, "synthetic:c1:256", "auto", "merge", "--iters", "20", "--gmres", "1e-5"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = [ln for ln in r.stdout.splitlines() if "iterations" in ln and "CONVERGED" in ln]
    assert len(lines) == 2, r.stdout
    assert "GMRES" in r.stdout
    its = [int(ln.split("]")[1].split()[0]) for ln in lines]
    assert all(i > 0 for i in its)
    mtx = tmp_path / "convdiff64.mtx"
    _write_mtx(mtx, *convdiff(64))
    r = subprocess.run([BIN, str(mtx), "auto", "--iters", "20", "--gmres", "1e-6", "--restart", "10", "--jacobi"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Jacobi" in r.stdout and "CONVERGED" in r.stdout
