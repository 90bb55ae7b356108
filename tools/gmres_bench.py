"""Where a restarted-GMRES step's time goes (spmvb200_gmres, csrc/gmres.cu), and what GMRES
costs against BiCGSTAB to a tolerance.

Matrix: the convection-diffusion form of lap2d at grid 2048 (4 M rows, fp64; A[i,i] += 1,
A[i,i-1] -= 1 for the west neighbour), b = A u with u seeded in [-1, 1], x0 = 0.  For restart 20
and 30, kinds merge and auto, M = I and Jacobi:
  - a solve capped at --steps Arnoldi steps (whole cycles), timed by the host clock around the
    call (which synchronises before it returns): ms per step, against one bare SpMV of that kind
    with SPMVB200_FLAG_STATIC_PATTERN timed by events;
  - a torch.profiler run of the same solve: the device time of the orthogonalisation kernels
    against the byte model below, as GB/s and % of the measured copy bandwidth (a
    device-to-device copy of 2 GiB, read + write) and of the data sheet (7.7 TB/s, HGX B200 at
    1000 W);
  - the same capped solve written in plain PyTorch (torch.sparse_csr_tensor matvec, CGS2 by
    tensor products, the Givens rotations on the host, one copy of h per step).
Then, per restart and M, the time to rtol 1e-8 with kind auto against spmvb200_bicgstab on the
same matrix (both capped at --cap steps or iterations).

Byte model of step j (k = j + 1 basis vectors), in vectors of n values, HBM traffic only:
  gmres_dot_kernel        read V, w                       k + 1
  gmres_orth_dot_kernel   read V, w, write w              k + 2  (its second read of V's
                                                                  lines is meant to hit the L2)
  gmres_orth_norm_kernel  read V, w, write w              k + 2
  gmres_scale_kernel      read w, write v                 2      (+ read dinv, write z: 4)
and once per cycle of k steps gmres_x_kernel, read V (k) and x, write x: k + 2 (+ dinv: k + 3).

    python tools/gmres_bench.py [--out FILE] [--quick]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from bicgstab_bench import convdiff  # noqa: E402
from cg_bench import DATASHEET_GBS, card, copy_gbs, events_ms, rhs  # noqa: E402
from spmv_samples_b200 import solve, spmv  # noqa: E402

ORTH = ("gmres_dot_kernel", "gmres_orth_dot_kernel", "gmres_orth_norm_kernel", "gmres_scale_kernel")


def orth_vectors(steps, m, jacobi):
    """Vectors each orthogonalisation kernel moves over `steps` steps in cycles of m."""
    out = dict.fromkeys(ORTH, 0)
    for s in range(steps):
        k = s % m + 1
        out["gmres_dot_kernel"] += k + 1
        out["gmres_orth_dot_kernel"] += k + 2
        out["gmres_orth_norm_kernel"] += k + 2
        out["gmres_scale_kernel"] += 4 if jacobi else 2
    return out


def profile_solve(m, b, kind, jacobi, restart, steps):
    from torch.profiler import ProfilerActivity, profile
    x = torch.zeros_like(b)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = solve.gmres(m.Ap, m.Aj, m.Ax, b, x, rtol=1e-14, restart=restart, max_iter=steps, kind=kind,
                          jacobi=jacobi)
        torch.cuda.synchronize()
    by_name = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        if t > 0:
            by_name[e.key] = by_name.get(e.key, 0.0) + t / 1e3
    return res, by_name


def torch_gmres(m, b, rtol, restart, max_iter, jacobi):
    """GMRES(restart) as a user would write it in PyTorch, right-preconditioned like the library."""
    A = torch.sparse_csr_tensor(m.Ap, m.Aj, m.Ax, size=(m.n_rows, m.n_cols))
    dinv = None
    if jacobi:
        rows = torch.repeat_interleave(torch.arange(m.n_rows, device="cuda"), torch.diff(m.Ap.long()))
        on_diag = m.Aj.long() == rows
        d = torch.zeros(m.n_rows, dtype=m.Ax.dtype, device="cuda")
        d.index_add_(0, rows[on_diag], m.Ax[on_diag])
        dinv = 1.0 / d
    n = b.numel()
    x = torch.zeros_like(b)
    tol = rtol * torch.linalg.vector_norm(b).item()
    V = torch.empty(restart + 1, n, dtype=b.dtype, device="cuda")
    it = 0
    while it < max_iter:
        r = b - A @ x
        beta = torch.linalg.vector_norm(r).item()
        if beta <= tol:
            break
        V[0] = r / beta
        R = [[0.0] * restart for _ in range(restart)]
        cs, sn, g = [0.0] * restart, [0.0] * restart, [beta] + [0.0] * restart
        k = 0
        for j in range(min(restart, max_iter - it)):
            w = A @ (V[j] * dinv if jacobi else V[j])
            h = V[:j + 1] @ w
            w -= V[:j + 1].T @ h
            h2 = V[:j + 1] @ w
            w -= V[:j + 1].T @ h2
            col = (h + h2).tolist()
            hn = torch.linalg.vector_norm(w).item()
            for i in range(j):
                col[i], col[i + 1] = cs[i] * col[i] + sn[i] * col[i + 1], -sn[i] * col[i] + cs[i] * col[i + 1]
            rr = math.hypot(col[j], hn)
            cs[j], sn[j] = (col[j] / rr, hn / rr) if rr else (1.0, 0.0)
            col[j] = rr
            g[j], g[j + 1] = cs[j] * g[j], -sn[j] * g[j]
            for i in range(j + 1):
                R[i][j] = col[i]
            it += 1
            k = j + 1
            if abs(g[j + 1]) <= tol or hn == 0.0:
                break
            V[j + 1] = w / hn
        y = [0.0] * k
        for i in range(k - 1, -1, -1):
            y[i] = (g[i] - sum(R[i][l] * y[l] for l in range(i + 1, k))) / R[i][i]
        u = torch.tensor(y, dtype=b.dtype, device="cuda") @ V[:k]
        x += u * dinv if jacobi else u
    return x, it


def timed(fn, reps=3):
    fn()   # warm
    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t0) * 1e3)
    return sorted(times)[len(times) // 2], out


def run_case(m, b, kind, jacobi, restart, steps, copy_bw):
    n, vb = m.n_rows, m.Ax.element_size()
    steps = steps // restart * restart   # whole cycles
    x = torch.zeros_like(b)

    def go():
        x.zero_()
        return solve.gmres(m.Ap, m.Aj, m.Ax, b, x, rtol=1e-14, restart=restart, max_iter=steps, kind=kind,
                           jacobi=jacobi)
    ms, res = timed(go)
    assert res.iterations == steps and not res.breakdown, res
    y = torch.empty_like(b)
    spmv.spmv_ex(kind, m.Ap, m.Aj, m.Ax, b, y)
    spmv_ms = events_ms(lambda: spmv.spmv_ex(kind, m.Ap, m.Aj, m.Ax, b, y, static_pattern=True), 200)
    _, by_name = profile_solve(m, b, kind, jacobi, restart, steps)
    model = orth_vectors(steps, restart, jacobi)
    kernels = {}
    for k, vecs in model.items():
        kms = sum(t for name, t in by_name.items() if k in name)
        gbs = vecs * n * vb / (kms * 1e-3) / 1e9 if kms > 0 else None
        kernels[k] = dict(us_per_step=round(kms * 1e3 / steps, 2), gbs=round(gbs, 1) if gbs else None,
                          pct_of_measured_copy=round(100 * gbs / copy_bw, 1) if gbs else None)
    orth_ms = sum(sum(t for name, t in by_name.items() if k in name) for k in ORTH)
    orth_bytes = sum(model.values()) * n * vb
    xk_ms = sum(t for name, t in by_name.items() if "gmres_x_kernel" in name)
    out = dict(case=m.name, kind=kind, jacobi=jacobi, restart=restart, dtype=str(m.Ax.dtype).replace("torch.", ""),
               n=n, nnz=m.nnz, steps=steps, solve_ms=round(ms, 3), ms_per_step=round(ms / steps, 5),
               bare_spmv_ms=round(spmv_ms, 5), orth_ms_per_step=round(orth_ms / steps, 5),
               orth_gbs=round(orth_bytes / (orth_ms * 1e-3) / 1e9, 1) if orth_ms else None,
               x_kernel_ms_per_cycle=round(xk_ms / (steps // restart), 5),
               device_busy_ms_per_step=round(sum(by_name.values()) / steps, 5),
               rel_residual=res.residual_norm / res.b_norm, kernels=kernels)
    if out["orth_gbs"]:
        out["orth_pct_of_measured_copy"] = round(100 * out["orth_gbs"] / copy_bw, 1)
        out["orth_pct_of_datasheet"] = round(100 * out["orth_gbs"] / DATASHEET_GBS, 1)
    tms, (_, it_t) = timed(lambda: torch_gmres(m, b, 1e-14, restart, steps, jacobi), reps=1)
    out.update(torch_steps=it_t, torch_ms_per_step=round(tms / max(it_t, 1), 5),
               speedup_per_step=round((tms / max(it_t, 1)) / (ms / steps), 2))
    return out


def to_tolerance(m, b, jacobi, restarts, cap):
    x = torch.zeros_like(b)
    out = dict(case=m.name, kind="auto", jacobi=jacobi, rtol=1e-8, cap=cap)

    def run(fn):
        x.zero_()
        return fn()
    for restart in restarts:
        ms, r = timed(lambda: run(lambda: solve.gmres(m.Ap, m.Aj, m.Ax, b, x, rtol=1e-8, restart=restart,
                                                      max_iter=cap, kind="auto", jacobi=jacobi)), reps=1)
        out[f"gmres{restart}"] = dict(ms=round(ms, 1), steps=r.iterations, converged=r.converged,
                                      rel_residual=r.residual_norm / r.b_norm)
    ms, r = timed(lambda: run(lambda: solve.bicgstab(m.Ap, m.Aj, m.Ax, b, x, rtol=1e-8, max_iter=cap, kind="auto",
                                                     jacobi=jacobi)), reps=1)
    out["bicgstab"] = dict(ms=round(ms, 1), iterations=r.iterations, converged=r.converged, breakdown=r.breakdown,
                           rel_residual=r.residual_norm / r.b_norm)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    ap.add_argument("--quick", action="store_true", help="small sizes only (a rehearsal)")
    ap.add_argument("--steps", type=int, default=240, help="Arnoldi steps per timed solve (whole cycles)")
    ap.add_argument("--cap", type=int, default=3000, help="step / iteration cap of the time-to-tolerance solves")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gmres_bench needs a CUDA device")
    torch.cuda.set_device(0)
    name, power = card()
    bw = copy_gbs()
    header = dict(card=name, power_limit_and_max_sm_clock=power, measured_copy_gbs=round(bw, 1),
                  datasheet_gbs=DATASHEET_GBS)
    print(json.dumps(header), flush=True)
    lines = [header]
    m = convdiff(256 if args.quick else 2048, torch.float64)
    b = rhs(m)
    for restart in (20, 30):
        for kind in ("merge", "auto"):
            for jacobi in (False, True):
                r = run_case(m, b, kind, jacobi, restart, args.steps, bw)
                print(json.dumps(r), flush=True)
                lines.append(r)
    for jacobi in (False, True):
        r = to_tolerance(m, b, jacobi, (20, 30), args.cap)
        print(json.dumps(r), flush=True)
        lines.append(r)
    if args.out:
        with open(args.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
