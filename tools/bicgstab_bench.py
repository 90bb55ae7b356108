"""Where a BiCGSTAB iteration's time goes (spmvb200_bicgstab, csrc/bicgstab.cu).

For each matrix, kind and preconditioner: one solve of A x = b (b = A u, u seeded in [-1, 1],
x0 = 0), timed by the host clock around the call (which synchronises before it returns); two
bare SpMVs of that kind with SPMVB200_FLAG_STATIC_PATTERN per iteration, timed by events; a
torch.profiler run of the solve for the device time of each of the five streaming kernels; and
the same solve written in plain PyTorch (torch.sparse_csr_tensor matvec, torch vector ops, one
.item() per convergence test, as tools/cg_bench.py's torch_cg does for CG).

Matrices: the convection-diffusion form of lap2d at grid 2048 (4 M rows, fp64; A[i,i] += 1,
A[i,i-1] -= 1 for the west neighbour), and R-MAT scale 20, edge factor 16, seed 3, fp32, made
strictly diagonally dominant (R + diag(1 + sum_k |R_ik|), duplicates summed) -- large enough
(18.2 M merge-path items) that kind merge builds the table plan and runs the persistent table
kernel for both SpMVs of every iteration.

Byte model per steady-state iteration (kept here, quoted in DESIGN.md), in vectors of n values:
  p kernel      read r p v, write p                          4   (+ read dinv, write p^: 6)
  rv kernel     read r^ v                                    2
  s kernel      read r v x p^, write s x                     6   (+ read dinv, write s^: 8)
  omega kernel  read t s                                     2
  r kernel      read s t r^ x, write r x                     6   (+ read s^: 7)
  total                                                      20  (Jacobi 25)
  SpMV          nnz*(4 + v) + (n+1)*o + 2*n*v, twice         (BASELINE.md section 3)
GB/s of each kernel = its bytes / its device time per iteration, against the measured copy
bandwidth (a device-to-device copy of 2 GiB, read + write) and the data sheet (7.7 TB/s for the
HGX B200, 1000 W), both labelled.

    python tools/bicgstab_bench.py [--out FILE] [--quick]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from cg_bench import DATASHEET_GBS, card, copy_gbs, events_ms, rhs  # noqa: E402
from spmv_samples_b200 import generate, solve, spmv  # noqa: E402

# kernel name -> vectors it moves per iteration, (without, with) Jacobi
KERNELS = {"bicgstab_p_kernel": (4, 6), "bicgstab_rv_kernel": (2, 2), "bicgstab_s_kernel": (6, 8),
           "bicgstab_omega_kernel": (2, 2), "bicgstab_r_kernel": (6, 7)}


def convdiff(grid, dtype):
    m = generate.lap2d(grid, dtype)
    rows = torch.repeat_interleave(torch.arange(m.n_rows, device="cuda"), torch.diff(m.Ap.long()))
    cols = m.Aj.long()
    m.Ax = m.Ax + (cols == rows).to(dtype) - (cols == rows - 1).to(dtype)
    m.name = f"convdiff_{grid}"
    return m


def rmat_dominant(scale, ef, seed, dtype):
    r = generate.rmat(scale, ef, seed, dtype)
    n = r.n_rows
    rows = torch.repeat_interleave(torch.arange(n, device="cuda"), torch.diff(r.Ap.long()))
    diag = 1.0 + torch.zeros(n, dtype=torch.float64, device="cuda").index_add_(0, rows, r.Ax.double().abs())
    keys = torch.cat([rows * n + r.Aj.long(), torch.arange(n, device="cuda") * (n + 1)])
    uk, inv = torch.unique(keys, sorted=True, return_inverse=True)
    vals = torch.zeros(uk.numel(), dtype=torch.float64, device="cuda").index_add_(0, inv, torch.cat([r.Ax.double(), diag]))
    Ap = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    Ap[1:] = torch.cumsum(torch.bincount(uk // n, minlength=n), 0)
    return generate.Csr(n, n, uk.numel(), Ap.int(), (uk % n).int(), vals.to(dtype), f"rmat_dominant_s{scale}")


def profile_solve(m, b, kind, jacobi, rtol, max_iter):
    """Device time per kernel name over one solve (torch.profiler, a run of its own)."""
    from torch.profiler import ProfilerActivity, profile
    x = torch.zeros_like(b)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = solve.bicgstab(m.Ap, m.Aj, m.Ax, b, x, rtol=rtol, max_iter=max_iter, kind=kind, jacobi=jacobi)
        torch.cuda.synchronize()
    by_name = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        if t > 0:
            by_name[e.key] = by_name.get(e.key, 0.0) + t / 1e3
    return res, by_name


def torch_bicgstab(m, b, rtol, max_iter, jacobi):
    """The solve a user would write, in scipy's order: torch sparse CSR matvec, vector ops,
    .item() for each convergence test."""
    A = torch.sparse_csr_tensor(m.Ap, m.Aj, m.Ax, size=(m.n_rows, m.n_cols))
    dinv = None
    if jacobi:
        rows = torch.repeat_interleave(torch.arange(m.n_rows, device="cuda"), torch.diff(m.Ap.long()))
        on_diag = m.Aj.long() == rows
        d = torch.zeros(m.n_rows, dtype=m.Ax.dtype, device="cuda")
        d.index_add_(0, rows[on_diag], m.Ax[on_diag])
        dinv = 1.0 / d
    x = torch.zeros_like(b)
    r = b - A @ x
    rh = r.clone()
    tol = rtol * torch.linalg.vector_norm(b).item()
    rho = torch.dot(rh, r)
    it = 0
    p = v = omega = alpha = None
    while it < max_iter:
        p = r.clone() if it == 0 else r + ((rho / rho_prev) * (alpha / omega)) * (p - omega * v)  # noqa: F821
        ph = p * dinv if jacobi else p
        v = A @ ph
        alpha = rho / torch.dot(rh, v)
        s = r - alpha * v
        x += alpha * ph
        it += 1
        if torch.linalg.vector_norm(s).item() <= tol:
            break
        sh = s * dinv if jacobi else s
        t = A @ sh
        omega = torch.dot(t, s) / torch.dot(t, t)
        x += omega * sh
        r = s - omega * t
        if torch.linalg.vector_norm(r).item() <= tol:
            break
        rho_prev, rho = rho, torch.dot(rh, r)
    return x, it


def run_case(m, kind, jacobi, rtol, max_iter, copy_bw):
    b = rhs(m)
    n, vb = m.n_rows, m.Ax.element_size()
    x = torch.zeros_like(b)
    res = solve.bicgstab(m.Ap, m.Aj, m.Ax, b, x, rtol=rtol, max_iter=max_iter, kind=kind, jacobi=jacobi)  # warm
    times = []
    for _ in range(3):
        x.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = solve.bicgstab(m.Ap, m.Aj, m.Ax, b, x, rtol=rtol, max_iter=max_iter, kind=kind, jacobi=jacobi)
        times.append((time.perf_counter() - t0) * 1e3)   # the call synchronises before it returns
    ms = sorted(times)[1]
    its = max(res.iterations, 1)
    # two bare SpMVs per iteration, static pattern, back to back
    y = torch.empty_like(b)
    spmv.spmv_ex(kind, m.Ap, m.Aj, m.Ax, b, y)
    spmv_ms = events_ms(lambda: spmv.spmv_ex(kind, m.Ap, m.Aj, m.Ax, b, y, static_pattern=True), 2 * its) * 2
    _, by_name = profile_solve(m, b, kind, jacobi, rtol, max_iter)
    kernels = {}
    for k, vecs in KERNELS.items():
        kms = sum(t for name, t in by_name.items() if k in name) / its
        gbs = vecs[jacobi] * n * vb / (kms * 1e-3) / 1e9 if kms > 0 else None
        kernels[k] = dict(us_per_iteration=round(kms * 1e3, 2), gbs=round(gbs, 1) if gbs else None,
                          pct_of_measured_copy=round(100 * gbs / copy_bw, 1) if gbs else None)
    k_ms = sum(v["us_per_iteration"] for v in kernels.values()) / 1e3
    vbytes = sum(v[jacobi] for v in KERNELS.values()) * n * vb
    all_ms = sum(by_name.values())
    out = dict(case=m.name, kind=kind, jacobi=jacobi, dtype=str(m.Ax.dtype).replace("torch.", ""), n=n, nnz=m.nnz,
               rtol=rtol, iterations=res.iterations, converged=res.converged, breakdown=res.breakdown,
               rel_residual=res.residual_norm / res.b_norm if res.b_norm else 0.0,
               solve_ms=round(ms, 3), ms_per_iteration=round(ms / its, 5),
               two_spmv_ms_per_iteration=round(spmv_ms, 5),
               five_kernels_ms_per_iteration=round(k_ms, 5),
               device_busy_ms_per_iteration=round(all_ms / its, 5),
               vector_bytes=vbytes, spmv_bytes=2 * m.algorithmic_bytes(),
               five_kernels_gbs=round(vbytes / (k_ms * 1e-3) / 1e9, 1) if k_ms > 0 else None,
               kernels=kernels)
    if out["five_kernels_gbs"]:
        out["five_kernels_pct_of_measured_copy"] = round(100 * out["five_kernels_gbs"] / copy_bw, 1)
        out["five_kernels_pct_of_datasheet"] = round(100 * out["five_kernels_gbs"] / DATASHEET_GBS, 1)
    torch_bicgstab(m, b, rtol, min(max_iter, 5), jacobi)  # warm
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _, it_t = torch_bicgstab(m, b, rtol, max_iter, jacobi)
    torch.cuda.synchronize()
    tms = (time.perf_counter() - t0) * 1e3
    out.update(torch_iterations=it_t, torch_ms=round(tms, 3), torch_ms_per_iteration=round(tms / max(it_t, 1), 5),
               speedup_per_iteration=round((tms / max(it_t, 1)) / (ms / its), 2))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    ap.add_argument("--quick", action="store_true", help="small sizes only (a rehearsal)")
    ap.add_argument("--max-iter", type=int, default=1000,
                    help="iteration cap (per-iteration cost is the point, not the count)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bicgstab_bench needs a CUDA device")
    torch.cuda.set_device(0)
    name, power = card()
    bw = copy_gbs()
    header = dict(card=name, power_limit_and_max_sm_clock=power, measured_copy_gbs=round(bw, 1),
                  datasheet_gbs=DATASHEET_GBS)
    print(json.dumps(header), flush=True)
    lines = [header]
    grid, scale = (256, 16) if args.quick else (2048, 20)
    cases = [
        (lambda: convdiff(grid, torch.float64), [("merge", False), ("auto", False), ("auto", True)], 1e-6),
        (lambda: rmat_dominant(scale, 16, 3, torch.float32), [("merge", False), ("merge", True)], 1e-6),
    ]
    for make, runs, rtol in cases:
        m = make()
        for kind, jacobi in runs:
            r = run_case(m, kind, jacobi, rtol, args.max_iter, bw)
            if kind == "merge":
                r["table_columns"] = spmv.hot_x_info(m.Aj)["table_columns"]
            print(json.dumps(r), flush=True)
            lines.append(r)
        del m
        spmv.release_cache()
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
