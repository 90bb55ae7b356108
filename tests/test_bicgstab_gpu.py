"""GPU suite for the BiCGSTAB solve (spmvb200_bicgstab through spmv_samples_b200.solve.bicgstab):
accuracy against the fp64 numpy restatement (tests/test_bicgstab_cpu.py), Jacobi, the table
plan of the merge kernel with x changing between the two SpMVs of an iteration, determinism,
exact early exit, edge cases, breakdown, the Jacobi diagonal check, the launch count, and
bin/spmv --bicgstab."""
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import cpu
from test_bicgstab_cpu import (bicgstab_reference, convdiff, jacobi_dinv, rmat_dominant, scaled_identity,
                               swap_pairs)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "bin", "spmv")
MAX_BATCH = 64   # kKrylovMaxBatch in csrc/krylov.cuh: iterations enqueued between two reads of the flags


@pytest.fixture(scope="module", autouse=True)
def _device(built_lib):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    torch.cuda.set_device(0)
    yield
    from spmv_samples_b200 import spmv
    spmv.release_cache()


_cache = {}


def problem(name, dtype=np.float64, offset=np.int32):
    """convdiff(grid) ("convdiff64") or rmat_dominant(scale) ("rmat14"), and b = A x_true for a
    seeded x_true in [-1, 1]: host arrays in the value type, plus their device copies."""
    key = (name, np.dtype(dtype).name, np.dtype(offset).name)
    if key not in _cache:
        size = int(name.replace("convdiff", "").replace("rmat", ""))
        Ap, Aj, Ax = convdiff(size, 1.0, np.float64, offset) if name.startswith("convdiff") \
            else rmat_dominant(size, 16, 3, np.float64, offset)
        Ax = Ax.astype(dtype)
        n = Ap.shape[0] - 1
        x_true = np.random.default_rng(size).uniform(-1.0, 1.0, n)
        b = cpu.spmv_fp64(Ap, Aj, Ax, x_true).astype(dtype)
        dev = tuple(torch.from_numpy(a).cuda() for a in (Ap, Aj, Ax, b))
        _cache[key] = (Ap, Aj, Ax, b, dev)
    return _cache[key]


def true_residual(Ap, Aj, Ax, b, x):
    return float(np.linalg.norm(b.astype(np.float64) - cpu.spmv_fp64(Ap, Aj, Ax, x.cpu().numpy())))


@pytest.mark.parametrize("kind", ["merge", "vector", "light", "stream", "auto"])
@pytest.mark.parametrize("offset", [np.int32, np.int64], ids=["o32", "o64"])
@pytest.mark.parametrize("grid", [64, 128])
def test_bicgstab_f64_accuracy(grid, offset, kind):
    from spmv_samples_b200 import solve
    rtol = 1e-8
    Ap, Aj, Ax, b, dev = problem(f"convdiff{grid}", np.float64, offset)
    res = solve.bicgstab(*dev, rtol=rtol, kind=kind)
    _, it_ref, conv_ref, _ = bicgstab_reference(Ap, Aj, Ax, b, rtol, Ap.shape[0] - 1)
    assert res.converged and not res.breakdown and conv_ref
    assert abs(res.iterations - it_ref) <= 2, (res.iterations, it_ref)
    bn = float(np.linalg.norm(b))
    assert res.b_norm == pytest.approx(bn, rel=1e-12)
    tr = true_residual(Ap, Aj, Ax, b, res.x)
    assert tr <= 1.01 * rtol * bn, (tr, rtol * bn)
    assert res.residual_norm == pytest.approx(tr, rel=1e-10)


@pytest.mark.parametrize("kind", ["merge", "auto"])
def test_bicgstab_f32(kind):
    from spmv_samples_b200 import solve
    rtol = 1e-4
    Ap, Aj, Ax, b, dev = problem("convdiff128", np.float32)
    res = solve.bicgstab(*dev, rtol=rtol, kind=kind)
    assert res.converged and not res.breakdown
    tr = true_residual(Ap, Aj, Ax, b, res.x)
    assert tr <= 2 * rtol * float(np.linalg.norm(b.astype(np.float64)))
    assert res.residual_norm == pytest.approx(tr, rel=1e-10)


def test_bicgstab_jacobi_on_rmat_dominant():
    from spmv_samples_b200 import solve
    rtol = 1e-10
    Ap, Aj, Ax, b, dev = problem("rmat14")
    plain = solve.bicgstab(*dev, rtol=rtol, kind="auto")
    jac = solve.bicgstab(*dev, rtol=rtol, kind="auto", jacobi=True)
    assert plain.converged and jac.converged
    assert jac.iterations < plain.iterations, (jac.iterations, plain.iterations)
    _, it_ref, _, _ = bicgstab_reference(Ap, Aj, Ax, b, rtol, Ap.shape[0] - 1, jacobi_dinv(Ap, Aj, Ax))
    assert abs(jac.iterations - it_ref) <= 2, (jac.iterations, it_ref)
    assert true_residual(Ap, Aj, Ax, b, jac.x) <= 1.01 * rtol * float(np.linalg.norm(b))


def test_bicgstab_on_the_table_plan():
    """R-MAT scale 20 in fp32 with kind merge: the static-pattern SpMVs build the table plan
    (csrc/hotx.cu) and the persistent table kernel runs both SpMVs of every iteration, on p^ and
    then on s^.  The solve is bit-identical to the one with the table off."""
    from spmv_samples_b200 import solve, spmv
    Ap, Aj, Ax = rmat_dominant(20, 16, 3, np.float32)
    n = Ap.shape[0] - 1
    # what makes the plan worth building, from the host matrix: 18.2 M merge-path items (at least
    # 4.8 M) and the 16 K most frequent columns take 54 % of the gathers (at least a tenth)
    counts = np.sort(np.bincount(Aj, minlength=n))[::-1]
    assert n + Aj.shape[0] >= 4_800_000 and counts[:16384].sum() >= 0.1 * Aj.shape[0]
    b = cpu.spmv_fp64(Ap, Aj, Ax, np.random.default_rng(20).uniform(-1.0, 1.0, n)).astype(np.float32)
    dev = [torch.from_numpy(a).cuda() for a in (Ap, Aj, Ax, b)]
    rtol = 1e-4
    spmv.release_cache()
    with_table = solve.bicgstab(*dev, rtol=rtol, kind="merge")
    info = spmv.hot_x_info(dev[1])
    assert info["table_columns"] > 0, info
    old = spmv.get_option("hot_x_table")
    spmv.set_option("hot_x_table", 0)
    try:
        spmv.release_cache()
        plain = solve.bicgstab(*dev, rtol=rtol, kind="merge")
        assert spmv.hot_x_info(dev[1])["table_columns"] == 0
    finally:
        spmv.set_option("hot_x_table", old)
        spmv.release_cache()
    assert with_table.converged and plain.converged
    assert with_table.iterations == plain.iterations
    assert with_table.residual_norm == plain.residual_norm
    assert torch.equal(with_table.x, plain.x)


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("kind", ["merge", "vector", "auto"])
def test_bicgstab_is_deterministic(kind, dtype):
    from spmv_samples_b200 import solve
    _, _, _, _, dev = problem("convdiff64", dtype)
    rtol = 1e-4 if dtype == np.float32 else 1e-8
    a = solve.bicgstab(*dev, rtol=rtol, kind=kind, jacobi=True)
    b = solve.bicgstab(*dev, rtol=rtol, kind=kind, jacobi=True)
    assert a.converged
    assert a.iterations == b.iterations and a.residual_norm == b.residual_norm
    assert torch.equal(a.x, b.x)


def test_bicgstab_early_exit_is_exact():
    """The flags stop every kernel of an iteration batch already enqueued: the solve that stops
    at m returns the same bits as one allowed exactly m iterations."""
    from spmv_samples_b200 import solve
    _, _, _, _, dev = problem("convdiff64")
    n = dev[0].numel() - 1
    full = solve.bicgstab(*dev, rtol=1e-8, kind="auto", max_iter=n)
    m = full.iterations
    assert full.converged and m > 10
    exact = solve.bicgstab(*dev, rtol=1e-8, kind="auto", max_iter=m)
    assert exact.converged and exact.iterations == m and torch.equal(exact.x, full.x)
    short = solve.bicgstab(*dev, rtol=1e-8, kind="auto", max_iter=m - 3)
    assert short.iterations == m - 3 and not short.converged and not short.breakdown


def test_bicgstab_edge_cases():
    from spmv_samples_b200 import solve
    Ap, Aj, Ax, b, dev = problem("convdiff32")
    dAp, dAj, dAx, db = dev
    n = Ap.shape[0] - 1
    # b = 0: x = 0 whatever x0 was
    res = solve.bicgstab(dAp, dAj, dAx, torch.zeros_like(db), torch.ones_like(db), rtol=1e-8)
    assert res.converged and res.iterations == 0 and res.b_norm == 0.0
    assert torch.count_nonzero(res.x) == 0
    # x0 already the solution (integer x: A x0 is exact)
    x0 = np.random.default_rng(5).integers(-3, 4, n).astype(np.float64)
    bx = torch.from_numpy(cpu.spmv_fp64(Ap, Aj, Ax, x0)).cuda()
    x = torch.from_numpy(x0).cuda()
    res = solve.bicgstab(dAp, dAj, dAx, bx, x, rtol=1e-8)
    assert res.converged and res.iterations == 0 and res.residual_norm == 0.0
    assert res.x is x and torch.equal(x.cpu(), torch.from_numpy(x0))
    # n = 0
    e = torch.zeros(0, dtype=torch.float64, device="cuda")
    res = solve.bicgstab(torch.zeros(1, dtype=torch.int32, device="cuda"),
                         torch.zeros(0, dtype=torch.int32, device="cuda"), e, e.clone())
    assert res.converged and res.iterations == 0 and res.x.numel() == 0
    # max_iter = 0: nothing moves, the residual is that of x0 = 0
    res = solve.bicgstab(*dev, rtol=1e-8, max_iter=0)
    assert not res.converged and not res.breakdown and res.iterations == 0
    assert torch.count_nonzero(res.x) == 0
    assert res.residual_norm == pytest.approx(float(np.linalg.norm(b)), rel=1e-12)


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
def test_bicgstab_breaks_down_on_swap_pairs(dtype):
    """(r^, v) = 0 exactly in the first iteration: a breakdown before x moves."""
    from spmv_samples_b200 import solve
    Ap, Aj, Ax = swap_pairs(1000, dtype)
    b = np.where(np.arange(2000) % 2 == 0, 1.0, 0.0).astype(dtype)
    res = solve.bicgstab(*[torch.from_numpy(a).cuda() for a in (Ap, Aj, Ax, b)], rtol=1e-8)
    assert res.breakdown and not res.converged and res.iterations == 0
    assert torch.count_nonzero(res.x) == 0


@pytest.mark.parametrize("jacobi", [False, True])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
def test_bicgstab_half_step_exit_on_4_identity(dtype, jacobi):
    """alpha = 1/4 exactly (1 with Jacobi), so s = 0: converged at the half step, one iteration,
    x = b / 4 bit for bit."""
    from spmv_samples_b200 import solve
    Ap, Aj, Ax = scaled_identity(5000, 4.0, dtype)
    b = np.random.default_rng(4).uniform(-1.0, 1.0, 5000).astype(dtype)
    res = solve.bicgstab(*[torch.from_numpy(a).cuda() for a in (Ap, Aj, Ax, b)], rtol=1e-8, jacobi=jacobi)
    assert res.converged and not res.breakdown and res.iterations == 1, res
    assert np.array_equal(res.x.cpu().numpy(), b / dtype(4))
    assert res.residual_norm == 0.0


@pytest.mark.parametrize("jacobi", [False, True])
@pytest.mark.parametrize("poison", ["nan_in_b", "inf_in_x0", "nan_off_diagonal"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
def test_bicgstab_non_finite_input_breaks_down_at_once(dtype, poison, jacobi):
    """A NaN or an inf present from the start makes ||r||^2 = rho (or ||b||) non-finite in the
    set-up: the solve reports a breakdown before the first iteration."""
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
    res = solve.bicgstab(dAp, dAj, dAx, db, x0, rtol=1e-6, jacobi=jacobi)
    assert res.breakdown and not res.converged and res.iterations == 0, res


def test_bicgstab_jacobi_rejects_a_bad_diagonal():
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
            solve.bicgstab(*d, rtol=1e-8, jacobi=True)
        assert e.value.status == 1
        assert solve.bicgstab(*d, rtol=1e-8, max_iter=3).iterations <= 3   # without Jacobi it runs


@pytest.mark.parametrize("kind", ["merge", "vector", "auto"])
def test_bicgstab_launch_count(kind):
    """Two SpMVs and five kernels per iteration; past the last one, at most one batch of
    iterations whose kernels return at once, plus the set-up and the final residual."""
    from spmv_samples_b200 import solve, spmv
    _, _, _, _, dev = problem("convdiff64")
    dAp, dAj, dAx, db = dev
    y = torch.empty_like(db)
    spmv.spmv_ex(kind, dAp, dAj, dAx, db, y)
    spmv.spmv_ex(kind, dAp, dAj, dAx, db, y, static_pattern=True)
    before = spmv.launch_count()
    spmv.spmv_ex(kind, dAp, dAj, dAx, db, y, static_pattern=True)
    per_spmv = spmv.launch_count() - before
    solve.bicgstab(*dev, rtol=1e-8, kind=kind)   # warm: statistics cache, scratch
    before = spmv.launch_count()
    res = solve.bicgstab(*dev, rtol=1e-8, kind=kind)
    launched = spmv.launch_count() - before
    assert res.converged
    per_it = 2 * per_spmv + 5
    assert launched >= res.iterations * per_it
    assert launched <= (res.iterations + MAX_BATCH) * per_it + 8, (launched, res.iterations, per_spmv)


def _write_mtx(path, Ap, Aj, Ax):
    n = Ap.shape[0] - 1
    rows = np.repeat(np.arange(n), np.diff(Ap))
    with open(path, "w") as f:
        f.write("%%MatrixMarket matrix coordinate real general\n")
        f.write(f"{n} {n} {Aj.shape[0]}\n")
        for i, j, v in zip(rows + 1, Aj.astype(np.int64) + 1, Ax):
            f.write(f"{i} {j} {float(v):.17g}\n")


def test_driver_bicgstab(tmp_path):
    if not os.path.exists(BIN):
        subprocess.run(["make", "-C", ROOT, "-s", "bin/spmv"], check=True)
    r = subprocess.run([BIN, "synthetic:c1:256", "auto", "merge", "--iters", "20", "--bicgstab", "1e-6"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = [ln for ln in r.stdout.splitlines() if "iterations" in ln and "CONVERGED" in ln]
    assert len(lines) == 2, r.stdout
    assert "BiCGSTAB" in r.stdout
    its = [int(ln.split("]")[1].split()[0]) for ln in lines]
    assert all(i > 0 for i in its)
    mtx = tmp_path / "convdiff64.mtx"
    _write_mtx(mtx, *convdiff(64))
    r = subprocess.run([BIN, str(mtx), "auto", "--iters", "20", "--bicgstab", "1e-6", "--jacobi"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Jacobi" in r.stdout and "CONVERGED" in r.stdout
