"""Where a conjugate-gradient iteration's time goes (spmvb200_cg, csrc/cg.cu).

For each matrix and kind: one solve of A x = b (b = A u, u seeded in [-1, 1], x0 = 0), timed by the
host clock around the call (which synchronises before it returns); the same number of bare SpMVs of that kind with
SPMVB200_FLAG_STATIC_PATTERN; a torch.profiler run of the solve for the device time of the three
CG kernels; and the same solve written in plain PyTorch (torch.sparse_csr_tensor matvec, torch
vector ops, one .item() per iteration for the convergence test) -- what a user would otherwise
write.

Byte model per iteration (kept here, quoted in DESIGN.md):
  SpMV     nnz*(4 + v) + (n+1)*o + 2*n*v        (BASELINE.md section 3: Aj, Ax, Ap, x, y)
  vectors  p.q 2n + update 6n (8n with Jacobi: + dinv read, z write) + direction 3n, times v
           (update: read x p r q, write x r; direction: read z p, write p)
GB/s of the CG kernels = vector bytes / their device time per iteration, against the measured
copy bandwidth (a device-to-device copy of 2 GiB, read + write) and the data sheet (7.7 TB/s for
the HGX B200, 1000 W), both labelled.

    python tools/cg_bench.py [--out FILE] [--quick]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from spmv_samples_b200 import generate, solve, spmv  # noqa: E402

DATASHEET_GBS = 7700.0
CG_KERNELS = ("cg_pq_kernel", "cg_update_kernel", "cg_direction_kernel")


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def events_ms(fn, reps=1):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def copy_gbs():
    src = torch.empty(1 << 31, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    dst.copy_(src)
    ms = min(events_ms(lambda: dst.copy_(src), 5) for _ in range(3))
    return 2 * src.numel() / (ms * 1e-3) / 1e9


def vector_bytes(n, vb, jacobi):
    return (2 + (8 if jacobi else 6) + 3) * n * vb


def spmv_bytes(m):
    return m.algorithmic_bytes()


def scaled_lap2d(grid, dtype, seed=7):
    """S A S with s in [1, 10]: the same pattern, a badly scaled diagonal."""
    m = generate.lap2d(grid, dtype)
    g = torch.Generator(device="cuda").manual_seed(seed)
    s = 1.0 + 9.0 * torch.rand(m.n_rows, generator=g, device="cuda", dtype=torch.float64)
    rows = torch.repeat_interleave(torch.arange(m.n_rows, device="cuda"), torch.diff(m.Ap.long()))
    m.Ax = (m.Ax.double() * s[rows] * s[m.Aj.long()]).to(dtype)
    m.name = f"lap2d_{grid}_scaled"
    return m


def rhs(m):
    u = generate.gen_x(m.n_cols, 11, m.Ax.dtype)
    b = torch.empty(m.n_rows, dtype=m.Ax.dtype, device="cuda")
    spmv.spmv_ex("merge", m.Ap, m.Aj, m.Ax, u, b)
    return b


def profile_cg(m, b, kind, jacobi, rtol, max_iter):
    """Device time per kernel name over one solve (torch.profiler, a run of its own)."""
    from torch.profiler import ProfilerActivity, profile
    x = torch.zeros_like(b)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = solve.cg(m.Ap, m.Aj, m.Ax, b, x, rtol=rtol, max_iter=max_iter, kind=kind, jacobi=jacobi)
        torch.cuda.synchronize()
    by_name = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        if t > 0:
            by_name[e.key] = (by_name.get(e.key, (0.0, 0))[0] + t / 1e3, e.count)
    return res, by_name


def torch_cg(m, b, rtol, max_iter, jacobi):
    """The solve a user would write: torch sparse CSR matvec, vector ops, .item() per iteration."""
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
    z = r * dinv if jacobi else r
    p = z.clone()
    rho = torch.dot(r, z)
    tol = rtol * torch.linalg.vector_norm(b).item()
    it = 0
    while it < max_iter:
        q = A @ p
        alpha = rho / torch.dot(p, q)
        x += alpha * p
        r -= alpha * q
        it += 1
        if torch.linalg.vector_norm(r).item() <= tol:
            break
        z = r * dinv if jacobi else r
        rz = torch.dot(r, z)
        p = z + (rz / rho) * p
        rho = rz
    return x, it


def run_case(name, m, kind, jacobi, rtol, max_iter, copy_bw, torch_baseline=True):
    b = rhs(m)
    n, vb = m.n_rows, m.Ax.element_size()
    x = torch.zeros_like(b)

    def one():
        x.zero_()
        return solve.cg(m.Ap, m.Aj, m.Ax, b, x, rtol=rtol, max_iter=max_iter, kind=kind, jacobi=jacobi)

    res = one()                       # warm: statistics, scratch, gather plans
    times = []
    for _ in range(3):
        x.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = solve.cg(m.Ap, m.Aj, m.Ax, b, x, rtol=rtol, max_iter=max_iter, kind=kind, jacobi=jacobi)
        times.append((time.perf_counter() - t0) * 1e3)   # the call synchronises before it returns
    ms = sorted(times)[1]
    its = max(res.iterations, 1)
    # the same number of bare SpMVs, static pattern, back to back
    y = torch.empty_like(b)
    spmv.spmv_ex(kind, m.Ap, m.Aj, m.Ax, b, y)
    spmv_ms = events_ms(lambda: spmv.spmv_ex(kind, m.Ap, m.Aj, m.Ax, b, y, static_pattern=True), its)
    # device time of the CG kernels
    _, by_name = profile_cg(m, b, kind, jacobi, rtol, max_iter)
    cg_ms = sum(t for k, (t, _) in by_name.items() if any(c in k for c in CG_KERNELS))
    all_ms = sum(t for t, _ in by_name.values())
    cg_per_it = cg_ms / its
    vbytes = vector_bytes(n, vb, jacobi)
    sbytes = spmv_bytes(m)
    out = dict(case=name, kind=kind, jacobi=jacobi, dtype=str(m.Ax.dtype).replace("torch.", ""), n=n, nnz=m.nnz,
               rtol=rtol, iterations=res.iterations, converged=res.converged,
               rel_residual=res.residual_norm / res.b_norm if res.b_norm else 0.0,
               solve_ms=round(ms, 3), ms_per_iteration=round(ms / its, 5),
               spmv_ms_per_iteration=round(spmv_ms, 5),
               cg_kernels_ms_per_iteration=round(cg_per_it, 5),
               device_busy_ms_per_iteration=round(all_ms / its, 5),
               non_kernel_share=round(max(0.0, 1.0 - (all_ms / its) / (ms / its)), 3),
               spmv_bytes=sbytes, vector_bytes=vbytes, vector_share_of_bytes=round(vbytes / (vbytes + sbytes), 3),
               cg_kernels_gbs=round(vbytes / (cg_per_it * 1e-3) / 1e9, 1) if cg_per_it > 0 else None)
    out["cg_kernels_pct_of_measured_copy"] = round(100 * out["cg_kernels_gbs"] / copy_bw, 1) if out["cg_kernels_gbs"] else None
    out["cg_kernels_pct_of_datasheet"] = round(100 * out["cg_kernels_gbs"] / DATASHEET_GBS, 1) if out["cg_kernels_gbs"] else None
    if torch_baseline:
        torch_cg(m, b, rtol, min(max_iter, 5), jacobi)  # warm
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        xt, it_t = torch_cg(m, b, rtol, max_iter, jacobi)
        torch.cuda.synchronize()
        tms = (time.perf_counter() - t0) * 1e3
        out.update(torch_iterations=it_t, torch_ms=round(tms, 3), torch_ms_per_iteration=round(tms / max(it_t, 1), 5),
                   speedup_per_iteration=round((tms / max(it_t, 1)) / (ms / its), 2))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    ap.add_argument("--quick", action="store_true", help="small grids only (a rehearsal)")
    ap.add_argument("--max-iter-4096", type=int, default=2000,
                    help="iteration cap of the 4096 grid (per-iteration cost is the point there)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("cg_bench needs a CUDA device")
    torch.cuda.set_device(0)
    name, power = card()
    bw = copy_gbs()
    header = dict(card=name, power_limit_and_max_sm_clock=power, measured_copy_gbs=round(bw, 1),
                  datasheet_gbs=DATASHEET_GBS)
    print(json.dumps(header), flush=True)
    lines = [header]
    g1, g2 = (128, 256) if args.quick else (1024, 4096)
    cases = [
        (f"lap2d_{g1}_f32", lambda: generate.lap2d(g1, torch.float32), ["merge", "vector", "auto"], False, 1e-6, None),
        (f"lap2d_{g1}_f64", lambda: generate.lap2d(g1, torch.float64), ["merge", "vector", "auto"], False, 1e-6, None),
        (f"lap2d_{g2}_f64", lambda: generate.lap2d(g2, torch.float64), ["auto"], False, 1e-6, args.max_iter_4096),
        (f"lap2d_{g1}_scaled_f64", lambda: scaled_lap2d(g1, torch.float64), ["auto"], None, 1e-6, None),
    ]
    for cname, make, kinds, jac, rtol, cap in cases:
        m = make()
        for kind in kinds:
            for jacobi in ((False, True) if jac is None else (jac,)):
                r = run_case(cname, m, kind, jacobi, rtol, cap or m.n_rows, bw)
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
