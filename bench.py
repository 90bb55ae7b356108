#!/usr/bin/env python
"""bench.py -- the contract benchmark.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload c5|c1..c4] [--kind auto|merge|vector|light]
                    [--exchange p2p|nccl] [--override SIZE] [--dump-outputs DIR]

Workload (BASELINE.json configs[4], the configuration the 1/2/4/8-GPU metric is quoted on):
R-MAT scale 27, edge factor 16 (134M rows, 2^31 nonzeros, int64 offsets, fp32), row-sharded
over N GPUs by nnz-balanced merge-path splits; a "step" is one power-iteration SpMV
x <- A x / ||A x|| over the whole matrix, including the exchange of the new x between GPUs.
The matrix (19.3 GB) fits one GPU, so N = 1 runs the same workload; total work is fixed as N
grows ("strong" scaling).

One JSON line on stdout (rank 0):
  value      whole-job GFLOP/s = 2 * nnz_total * K / t, t = CUDA-event time of K steps, max over
             ranks, inputs resident in HBM
  gbs        the same as effective GB/s on the algorithmic byte count
  e2e        the same metric through the host-buffer API (CsrMatrix.spmv): x from pinned host
             memory to the device, kernel, y back to the host, every step
  roofline   dominant kernel (rank 0): algorithmic bytes of its launch / its CUDA-event duration,
             against the measured HBM copy bandwidth in MEASURED_PEAKS.json
  cpu_baseline  the reference's CPU CSR loop (oracle/_ref when built, else the oracle port) on
             the host cores, on a bounded row sample of the same matrix

`--impl reference` times that CPU path alone (rank 0 only) and prints the same line with
"impl": "reference".

`--dump-outputs DIR` (own arm) writes, after the timed steps, what a caller of the power
iteration receives from the last of them: DIR/x.npy (the iterate A x, not yet divided by its
norm; a fixed seeded sample when it is larger than 32 MB) and DIR/eigen_estimate.npy (||A x||).
The matrix and x0 are fixed by the seed, so two builds run with the same arguments can be
compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "SpMV GFLOP/s and achieved HBM GB/s vs roofline at 1/2/4/8 B200"
UNIT = "GFLOP/s"
SEED = 0x5EEDB200


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=100)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--workload", default="c5", choices=["c1", "c2", "c3", "c4", "c5"])
    p.add_argument("--override", type=int, default=0,
                   help="shrink the workload (R-MAT scale / rows / grid); development only")
    p.add_argument("--kind", default="auto")
    p.add_argument("--exchange", default="auto", choices=["auto", "mc", "p2p", "nccl"])
    p.add_argument("--row-weight", default="1/1",
                   help="multi-GPU row split: cost of a row in nonzeros, num/den (1/1 = merge path)")
    p.add_argument("--rebalance", type=int, default=2,
                   help="multi-GPU: rounds of re-splitting the rows from measured per-rank local "
                        "step times (partition + tile kernel + fix-up + norm) before the timed region")
    p.add_argument("--e2e-steps", type=int, default=24)
    p.add_argument("--e2e-slots", type=int, default=0, choices=[0, 1, 2, 3, 4],
                   help="host-buffer calls in flight in the e2e leg (own stream + device x/y each); "
                        "0 = 4 on one GPU (measured: 20.6 / 12.5 / 12.0 ms per step with 2 / 3 / 4), 3 on several")
    p.add_argument("--cpu-seconds", type=float, default=15.0,
                   help="budget of the cpu_baseline leg (own arm)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--opts", default="", help="library options name=value,... (experiments; recorded in config)")
    p.add_argument("--no-configs", action="store_true",
                   help="skip the c1..c4 + cuSPARSE leg (N = 1 only; outside the timed region)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write the iterate x and the eigenvalue estimate as "
                        "DIR/<name>.npy (own arm, rank 0)")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        p.error("--dump-outputs writes the own arm's outputs; the reference arm has none")
    return args


def measured_peak():
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def kernel_source_sha():
    """sha1 over the sources of the dominant kernels: a traffic figure captured under ncu is only
    quoted while the kernel it was captured from is the kernel that ran."""
    import hashlib
    h = hashlib.sha1()
    for f in ("merge.cu", "hotx.cu", "common.cuh", "vector.cu", "stream.cu", "light.cu", "row_dot.cuh"):
        try:
            h.update(open(os.path.join(ROOT, "spmv_samples_b200", "csrc", f), "rb").read())
        except OSError:
            pass
    return h.hexdigest()[:16]


def traffic_lookup(workload_key, kernel):
    """DRAM bytes per launch of `kernel` on `workload_key` from profiles/traffic.json (one
    `ncu --set full` capture each), or None when the capture belongs to another kernel or to
    an older version of the kernel sources."""
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return None, "profiles/traffic.json missing"
    sha = kernel_source_sha()
    for e in tj.get("captures", []):
        if e.get("workload") == workload_key and e.get("kernel") == kernel:
            if e.get("kernel_source_sha") == sha:
                return e.get("dram_bytes"), e.get("source")
            return None, (f"capture of {kernel} exists ({e.get('source')}) but predates the current "
                          f"kernel sources (sha {e.get('kernel_source_sha')} vs {sha}): not quoted")
    return None, f"no capture of {kernel} on {workload_key}"


def workload_desc(name, override):
    from spmv_samples_b200 import generate
    d = generate.CONFIGS[name]["desc"]
    return d + (f" [override {override}]" if override else "")


# --------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """SM clock, max clock and throttle reasons of one GPU, sampled during the timed region."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
               0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown"}

    def __init__(self, index, period=0.01):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self._halt.is_set():
            try:
                self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                try:
                    r = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    r = int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def finish(self):
        self._halt.set()
        if self.is_alive():
            self.join(timeout=1.0)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# --------------------------------------------------------------------------- CPU leg
def build_row_sample(m, sample_nnz_target, n_blocks=16):
    """16 equally spaced blocks of consecutive rows of the workload matrix, concatenated into one
    CSR on the host (offsets rebased to 0, which changes no arithmetic)."""
    import numpy as np
    import torch

    per_block = max(1, sample_nnz_target // n_blocks)
    Ap_full = m.Ap
    pieces_Ap, pieces_Aj, pieces_Ax = [np.zeros(1, dtype=np.int64)], [], []
    base = 0
    rows_total = 0
    for b in range(n_blocks):
        r0 = (m.n_rows * b) // n_blocks
        r_hi = (m.n_rows * (b + 1)) // n_blocks
        if r_hi <= r0:
            continue
        k0 = int(Ap_full[r0].item())
        target = torch.tensor([k0 + per_block], device=Ap_full.device, dtype=Ap_full.dtype)
        r1 = int(torch.searchsorted(Ap_full[r0:r_hi + 1], target, right=True).item()) - 1 + r0
        r1 = max(r0 + 1, min(r1, r_hi))
        k1 = int(Ap_full[r1].item())
        pieces_Ap.append((Ap_full[r0 + 1:r1 + 1].to(torch.int64) - k0 + base).cpu().numpy())
        pieces_Aj.append(m.Aj[k0:k1].cpu().numpy())
        pieces_Ax.append(m.Ax[k0:k1].cpu().numpy())
        base += k1 - k0
        rows_total += r1 - r0
    Ap = np.concatenate(pieces_Ap)
    Aj = np.ascontiguousarray(np.concatenate(pieces_Aj))
    Ax = np.ascontiguousarray(np.concatenate(pieces_Ax))
    if m.Ap.dtype == torch.int32:
        Ap = Ap.astype(np.int32)
    return Ap, Aj, Ax, rows_total


def time_cpu_reference(Ap, Aj, Ax, x, rows_total, steps, warmup, seconds_budget):
    """Time the reference's CPU CSR loop on a host CSR sample, all host threads, for exactly
    `steps` timed calls after `warmup`.  If warmup + steps calls would not fit the time budget the
    sample is cut to a prefix of its rows (x stays full length, so the gathers miss the CPU caches
    the way the full problem's do).  Returns (gflops, info dict)."""
    import numpy as np

    from oracle import cpu

    threads = os.cpu_count() or 1
    total = warmup + steps
    use_ref = cpu.have_ref() and not (Ap.dtype == np.int64 and Ax.dtype == np.float64)
    rows_all, nnz_all = rows_total, int(Ap[-1])

    def runner(Ap_, Aj_, Ax_):
        return (lambda: cpu.ref_spmv_mt(Ap_, Aj_, Ax_, x, threads)) if use_ref else \
               (lambda: cpu.spmv_mt(Ap_, Aj_, Ax_, x, threads))

    run = runner(Ap, Aj, Ax)
    while True:
        run()                                 # first touch
        t0 = time.perf_counter()
        _, used = run()                       # calibration
        t_one = time.perf_counter() - t0
        nnz_s = int(Ap[-1])
        if t_one * total <= seconds_budget or nnz_s <= (1 << 20):
            break
        keep = max(1 << 20, int(nnz_s * seconds_budget / (t_one * total) * 0.8))
        r = max(1, int(np.searchsorted(Ap, keep, side="right")) - 1)
        Ap = np.ascontiguousarray(Ap[:r + 1])
        Aj, Ax = Aj[:int(Ap[-1])], Ax[:int(Ap[-1])]
        rows_total = r
        run = runner(Ap, Aj, Ax)
    for _ in range(max(0, warmup - 2)):
        run()
    t0 = time.perf_counter()
    for _ in range(steps):
        run()
    dt = (time.perf_counter() - t0) / steps
    # the reference as shipped is single threaded: time that too, once
    t0 = time.perf_counter()
    if use_ref:
        cpu.ref_spmv(Ap, Aj, Ax, x)
    else:
        cpu.spmv(Ap, Aj, Ax, x)
    dt1 = time.perf_counter() - t0
    info = {
        "kind": "reference" if use_ref else "port",
        "cores": int(used),
        "host_cores": int(threads),
        "sample": f"{rows_total} rows / {nnz_s} nonzeros"
                  + (f" (cut from {rows_all} / {nnz_all} to fit the time budget)" if nnz_s != nnz_all else "")
                  + " in equally spaced row blocks of the workload matrix, full-length x, "
                  f"{steps} timed calls of "
                  + ("reference SpMV_cpu_navie (oracle/_ref) on row blocks from all host threads"
                     if use_ref else "the oracle port of SpMV_cpu_navie, row blocks on all host threads"),
        "sample_rows": int(rows_total), "sample_nnz": int(nnz_s),
        "single_thread_value": 2.0 * nnz_s / dt1 / 1e9,
        "steps": steps,
        "ms_per_step": dt * 1e3,
    }
    return 2.0 * nnz_s / dt / 1e9, info


def cpu_reference_leg(global_csr, x_dev, steps, warmup, seconds_budget, sample_nnz_target=1 << 26):
    """cpu_baseline leg of the own arm: sample the resident matrix, time the reference on it."""
    Ap, Aj, Ax, rows_total = build_row_sample(global_csr, sample_nnz_target)
    return time_cpu_reference(Ap, Aj, Ax, x_dev.cpu().numpy(), rows_total, steps, warmup, seconds_budget)


# --------------------------------------------------------------------------- reference arm
SAMPLER_SCRIPT = r"""
import sys, numpy as np, torch
sys.path.insert(0, {root!r})
import bench
from spmv_samples_b200 import generate
torch.cuda.set_device(0)
m = generate.make_config({workload!r}, bench.SEED, scale_override={override!r})
x = generate.gen_x(m.n_cols, bench.SEED, m.Ax.dtype)
Ap, Aj, Ax, rows = bench.build_row_sample(m, {target}, n_blocks=64)
np.save({out!r} + "/Ap.npy", Ap); np.save({out!r} + "/Aj.npy", Aj); np.save({out!r} + "/Ax.npy", Ax)
np.save({out!r} + "/x.npy", x.cpu().numpy())
np.save({out!r} + "/meta.npy", np.array([rows, m.n_rows, m.nnz, m.Ap.element_size() * 8, m.algorithmic_bytes()], dtype=np.int64))
"""


def sample_in_subprocess(args, target_nnz):
    """The workload's matrix only exists as a device generator (csrc/gen.cu); the reference arm must
    not have this repository's library in the process it times.  So a child process generates the
    matrix on the GPU, cuts the row sample and leaves it on disk; the timed process only ever loads
    numpy arrays and oracle/_ref."""
    import subprocess
    import tempfile

    import numpy as np
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    out = tempfile.mkdtemp(prefix="spmv_ref_sample_", dir=base)
    code = SAMPLER_SCRIPT.format(root=ROOT, workload=args.workload, override=(args.override or None),
                                 target=int(target_nnz), out=out)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
    if r.returncode != 0:
        raise RuntimeError("sampler subprocess failed: " + (r.stderr or "")[-400:])
    arrs = {k: np.load(os.path.join(out, k + ".npy")) for k in ("Ap", "Aj", "Ax", "x", "meta")}
    import shutil
    shutil.rmtree(out, ignore_errors=True)
    return arrs


def reference_arm(args, rank, world):
    if rank != 0:
        return 0
    line = {"impl": "reference", "metric": METRIC, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic"}
    have_gpu = False
    try:
        # asked of a child process: it honours CUDA_VISIBLE_DEVICES as the sampler will, and this
        # process never creates a CUDA context
        import subprocess
        probe = "import sys, torch; sys.exit(0 if torch.cuda.is_available() else 1)"
        have_gpu = subprocess.run([sys.executable, "-c", probe], capture_output=True, timeout=300).returncode == 0
    except Exception:
        have_gpu = False
    note = None
    if have_gpu:
        # 2^28 nonzeros = 12.5 % of the workload's 2^31, in 64 equally spaced row blocks
        a = sample_in_subprocess(args, 1 << 28)
        Ap, Aj, Ax, x = a["Ap"], a["Aj"], a["Ax"], a["x"]
        rows_s, n_rows, nnz, off_bits, alg_bytes = (int(v) for v in a["meta"])
    else:
        # no GPU, no device generator: the host restatement at a scale the host can build
        import numpy as np

        from oracle import generators as g
        scale = 20
        Ap, Aj, Ax = g.rmat(scale, 16, SEED, offset_dtype=np.int64)
        x = g.gen_x(SEED, 1 << scale)
        rows_s, n_rows, nnz, off_bits = 1 << scale, 1 << scale, int(Ap[-1]), 64
        alg_bytes = nnz * 8 + (n_rows + 1) * 8 + n_rows * 8
        note = f"no GPU: R-MAT scale {scale} generated on the host instead of the workload"
    value, info = time_cpu_reference(Ap, Aj, Ax, x, rows_s, args.steps, args.warmup, seconds_budget=150.0)
    info["value"] = value
    info["unit"] = UNIT
    info["sample_fraction_of_nnz"] = info["sample_nnz"] / max(nnz, 1)
    line.update({
        "value": value,
        "ms_per_step": info["ms_per_step"],
        "steps": info["steps"],
        "config": {"workload": workload_desc(args.workload, args.override), "seed": SEED,
                   "rows": n_rows, "nnz": nnz, "offset_bits": off_bits,
                   "algorithmic_bytes_per_spmv": alg_bytes,
                   "step": "one CPU CSR SpMV (reference SpMV_cpu_navie) over a bounded row sample of the "
                           "workload matrix; GFLOP/s = 2 * sample nnz / time, a rate comparable with the "
                           "own arm's 2 * nnz / time",
                   "kind": "reference/include/spmv/cpu_navie.hpp:3-17 compiled by oracle/Makefile",
                   "sample_fraction_of_nnz": info["sample_fraction_of_nnz"],
                   "process": "this process never loads libspmvb200.so: a child process generated the "
                              "matrix and cut the sample" if have_gpu else "host-generated sample",
                   "note": note},
        "cpu_baseline": info,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })
    print(json.dumps(line), flush=True)
    return 0


# --------------------------------------------------------------------------- parity leg
TOL = {4: 1e-5, 8: 1e-13}   # |y - y_ref| <= tol * sum_j |a_ij x_j| per row (BASELINE.json north_star)


def parity_leg(csr, x, y, n_random=3000, n_heavy=6, seed=0):
    """Checker, outside every timed region: y (device, one plain SpMV of `csr`) against the fp64
    oracle on a row sample -- the `n_heavy` longest rows, `n_random` random rows, the first and the
    last -- gathered into a sub-CSR on the device and evaluated on the host by oracle.cpu
    (the restatement of reference/include/spmv/cpu_navie.hpp:3-35, pinned to oracle/_ref)."""
    import numpy as np
    import torch

    from oracle import cpu

    if csr.n_rows == 0:
        return {"rows_sampled": 0, "max_err_over_scale": 0.0, "tol": None, "ok": True}
    lens = csr.Ap[1:] - csr.Ap[:-1]
    heavy = torch.topk(lens, min(n_heavy, csr.n_rows)).indices
    gen = torch.Generator(device="cuda").manual_seed(seed)
    rnd = torch.randint(0, csr.n_rows, (n_random,), device="cuda", generator=gen)
    rows = torch.unique(torch.cat([heavy, rnd, torch.tensor([0, csr.n_rows - 1], device="cuda")]))
    starts, ends = csr.Ap[rows].long(), csr.Ap[rows + 1].long()
    seg = ends - starts
    sub_Ap = torch.zeros(rows.numel() + 1, dtype=torch.int64, device="cuda")
    sub_Ap[1:] = torch.cumsum(seg, 0)
    total = int(sub_Ap[-1])
    pos = torch.arange(total, device="cuda") - torch.repeat_interleave(sub_Ap[:-1], seg) \
        + torch.repeat_interleave(starts, seg)
    Aj, Ax, Ap = csr.Aj[pos].cpu().numpy(), csr.Ax[pos].cpu().numpy(), sub_Ap.cpu().numpy()
    xh = x.cpu().numpy()
    y64 = cpu.spmv_fp64(Ap, Aj, Ax, xh)
    scale = cpu.abs_scale(Ap, Aj, Ax, xh)
    got = y[rows].cpu().numpy().astype(np.float64)
    tol = TOL[csr.Ax.element_size()]
    err = np.abs(got - y64)
    nz = scale > 0
    ratio = float((err[nz] / scale[nz]).max()) if nz.any() else 0.0
    ok = bool(np.all(err <= tol * scale))
    return {"rows_sampled": int(rows.numel()), "nnz_sampled": total, "max_err_over_scale": ratio,
            "tol": tol, "ok": ok,
            "oracle": "oracle.cpu.spmv_fp64 (fp64 restatement of cpu_navie.hpp:3-17) on the "
                      f"{n_heavy} longest rows + {n_random} random rows + first + last"}


# --------------------------------------------------------------------------- configs leg
def _median_us(fn, flush, iters):
    import torch
    ts = []
    for _ in range(iters):
        flush.zero_()            # L2 flushed: 512 MB written between timed calls
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


def configs_leg(peak, iters=15):
    """c1..c4 of BASELINE.json at full size, one GPU: every kind of this library and cuSPARSE
    (setup hoisted; ALG_DEFAULT as the reference calls it, cusparse.cuh:76-78, then with
    cusparseSpMV_preprocess, then CSR_ALG2), CUDA events around single calls with the L2 flushed in
    between, median; the selector's choice; a same-size device copy and the pure-gather yardstick;
    parity of the selected kernel on sampled rows.  Outside the timed region of the headline."""
    import torch

    from spmv_samples_b200 import generate, spmv
    kind_names = {0: "merge", 1: "vector", 2: "light", 3: "auto", 4: "cusparse", 5: "stream"}
    spmv.set_option("time_main_kernel", 0)   # the per-kernel event pair costs ~5 us per call: headline leg only
    flush = torch.empty(512 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")
    out = {}
    yard = {}
    for cfg in ("c1", "c2", "c3", "c4"):
        m = generate.make_config(cfg, SEED)
        x = generate.gen_x(m.n_cols, SEED, m.Ax.dtype)
        y = torch.empty(m.n_rows, dtype=m.Ax.dtype, device="cuda")
        st = spmv.row_stats(m.Ap, nnz=m.nnz)
        alg = m.algorithmic_bytes()
        call = lambda k: spmv.SpMV(k, m.n_rows, m.n_cols, m.nnz, m.Ap, m.Aj, m.Ax, x, y)
        ours = {}
        # "stream" gives a row to a thread: only timed on the matrices it is meant for (a hub row
        # of R-MAT scale 24 keeps one thread busy for a second)
        kinds = ["merge", "vector", "light", "auto"]
        if st["mean_row_len"] <= 8.0 and st["max_row_len"] <= 64:   # wider than the selector's own rule (<= 6)
            kinds.insert(3, "stream")
        for k in kinds:
            for _ in range(3):
                call(k)
            ours[k] = round(_median_us(lambda: call(k), flush, iters), 2)
        best = min((k for k in kinds if k != "auto"), key=lambda k: ours[k])
        # the same calls from a caller that vouches for an unchanged matrix (the flag of
        # spmvb200_spmv; here through option "assume_static_pattern"): the merge-path partition is
        # reused and, on a skewed column distribution, the hot-x / table plan is built (warm-up) and used
        spmv.set_option("assume_static_pattern", 1)
        static = {}
        for k in ("merge", "auto"):
            for _ in range(3):
                call(k)
            static[k] = round(_median_us(lambda: call(k), flush, iters), 2)
        hx = spmv.hot_x_info(m.Aj)
        spmv.set_option("assume_static_pattern", 0)
        spmv.release_cache()
        call("auto")
        torch.cuda.synchronize()
        par = parity_leg(m, x, y)
        cus = {}
        for label, opts in (("alg_default", {"cusparse_alg": 0, "cusparse_preprocess": 0}),
                            ("alg_default_preprocess", {"cusparse_alg": 0, "cusparse_preprocess": 1}),
                            ("csr_alg2", {"cusparse_alg": 2, "cusparse_preprocess": 0})):
            try:
                for name, v in opts.items():
                    spmv.set_option(name, v)
                for _ in range(3):
                    call("cusparse")
                cus[label] = round(_median_us(lambda: call("cusparse"), flush, iters), 2)
            except Exception as e:   # the baseline is reported, never required
                cus[label] = None
                cus[label + "_error"] = str(e)[:120]
        spmv.set_option("cusparse_alg", 0)
        spmv.set_option("cusparse_preprocess", 0)
        half = alg // 8
        src = torch.empty(half, dtype=torch.float32, device="cuda")
        dst = torch.empty_like(src)
        copy_us = _median_us(lambda: dst.copy_(src), flush, iters)
        del src, dst
        t_auto = ours["auto"] * 1e-6
        entry = {
            "desc": generate.CONFIGS[cfg]["desc"], "rows": m.n_rows, "nnz": m.nnz,
            "algorithmic_bytes": alg, "selected_kernel": kind_names.get(st["chosen_kind"]),
            "us": ours, "best_kind": best,
            "us_static_pattern": static,
            "static_pattern_plan": {"hot_columns": hx["hot_columns"], "hot_share": round(hx["hot_share"], 4),
                                    "table_columns": hx["table_columns"], "table_share": round(hx["table_share"], 4)},
            "frac_static_pattern": alg / (static["auto"] * 1e-6) / 1e9 / peak,
            "auto_gbs": alg / t_auto / 1e9, "auto_gflops": m.flops() / t_auto / 1e9,
            "frac": alg / t_auto / 1e9 / peak, "frac_of_datasheet_8000": alg / t_auto / 1e9 / 8000.0,
            "cusparse_us": cus, "copy_same_bytes_us": round(copy_us, 2),
            "parity": par,
        }
        best_cus = min([v for k, v in cus.items() if isinstance(v, float)], default=None)
        entry["auto_over_best_cusparse"] = (best_cus / ours["auto"]) if best_cus else None
        if cfg in ("c2", "c3"):
            key = m.n_cols
            if key not in yard:
                yard[key] = spmv.gather_yardstick(m.n_cols)
            entry["gather_yardstick_ggathers_s"] = yard[key]
            entry["auto_ggathers_s"] = m.nnz / t_auto / 1e9
        out[cfg] = entry
        spmv.release_cache()
        del m, x, y
        torch.cuda.empty_cache()
    out["_method"] = ("CUDA events around one call, L2 flushed (512 MB written) before each, median of "
                      f"{iters}; cuSPARSE handle / descriptors / buffer created once outside the timing")
    del flush
    torch.cuda.empty_cache()
    return out


# --------------------------------------------------------------------------- outputs
DUMP_X_BYTES = 32 << 20


def dump_outputs(out_dir, x, eigen_estimate):
    """--dump-outputs: x (PowerIteration.current_x, in its own dtype) and ||A x|| as .npy files.
    An x of more than DUMP_X_BYTES is sampled: one entry from each of k equal strata of its index
    range at a seeded offset, so every run on the same matrix size writes the same entries."""
    import numpy as np
    import torch

    n, k = x.numel(), DUMP_X_BYTES // x.element_size()
    if n > k:
        lo = np.arange(k, dtype=np.int64) * n // k
        width = np.diff(np.append(lo, n))
        idx = lo + (np.random.default_rng(SEED).random(k) * width).astype(np.int64)
        x = x[torch.from_numpy(idx).to(x.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "x.npy"), x.cpu().numpy())
    np.save(os.path.join(out_dir, "eigen_estimate.npy"), np.array([eigen_estimate], dtype=np.float64))


# --------------------------------------------------------------------------- own arm
def own_arm(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist

    from spmv_samples_b200 import _lib, generate, spmv
    from spmv_samples_b200.dist import PowerIteration, shard_rows
    from spmv_samples_b200.matrix import CsrMatrix

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path "
                         "(use --impl reference for the CPU baseline)")
    _lib.lib()
    # diagnostics only (the contract line needs both): BENCH_NO_KTIMER=1 leaves the per-kernel
    # event timer off, BENCH_NO_SAMPLER=1 the NVML clock sampler
    spmv.set_option("time_main_kernel", 0 if os.environ.get("BENCH_NO_KTIMER") else 1)
    for kv in filter(None, args.opts.split(",")):
        name, v = kv.split("=")
        spmv.set_option(name, int(v))
    peak, peak_src = measured_peak()

    # ---- the matrix: every rank builds the global CSR on its own GPU, keeps its rows
    t_gen = time.perf_counter()
    gm = generate.make_config(args.workload, SEED, scale_override=args.override or None)
    n, n_cols, nnz_total = gm.n_rows, gm.n_cols, gm.nnz
    if n != n_cols:
        raise SystemExit("power iteration needs a square matrix")
    alg_bytes_total = gm.algorithmic_bytes()
    stats = spmv.row_stats(gm.Ap, nnz=gm.nnz)
    weight = tuple(int(v) for v in args.row_weight.split("/"))
    shard = shard_rows(gm, rank, world, weight=weight)
    x_for_cpu = generate.gen_x(n_cols, SEED, gm.Ax.dtype) if (rank == 0 and world == 1) else None
    cpu_info = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            v, cpu_info = cpu_reference_leg(gm, x_for_cpu, steps=3, warmup=1,
                                            seconds_budget=args.cpu_seconds)
            cpu_info["value"] = v
            cpu_info["unit"] = UNIT
        except Exception as e:  # the baseline is reported, never required
            cpu_info = {"value": None, "unit": UNIT, "cores": 0, "kind": "port",
                        "sample": f"failed: {e}"}
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t_gen

    it = PowerIteration(shard, n, kind=args.kind, exchange=args.exchange)
    rebalance_log = []
    if world > 1:
        for _ in range(args.rebalance):
            for _ in range(3):
                it.step()
            times, rb = it.rebalance(gm, steps=5, weight=weight)
            rebalance_log.append({"local_ms_before": [round(v, 4) for v in times], "row_bounds": rb})
        shard = it.shard
        del gm
        torch.cuda.empty_cache()
    local = shard.csr

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up, then K timed steps between barriers, CUDA events, max over ranks
    for _ in range(max(args.warmup, 3)):
        it.step()
    barrier()
    d_ms, d_n = C_double(), C_int64()
    import ctypes
    _lib.lib().spmvb200_main_kernel_time(ctypes.byref(d_ms), ctypes.byref(d_n))   # reset the kernel timer
    launches0 = spmv.launch_count()
    sampler = ClockSampler(physical_gpu_index(local_rank))
    if os.environ.get("BENCH_NO_SAMPLER"):
        sampler.ok = False
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        it.step()
    e1.record()
    barrier()
    clocks = sampler.finish()
    elapsed_ms = e0.elapsed_time(e1)
    launches = spmv.launch_count() - launches0
    _lib.lib().spmvb200_main_kernel_time(ctypes.byref(d_ms), ctypes.byref(d_n))
    kern_ms = d_ms.value / max(d_n.value, 1)
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device="cuda")
    per_rank = torch.zeros(world, 3, dtype=torch.float64, device="cuda")
    per_rank[rank, 0], per_rank[rank, 1], per_rank[rank, 2] = kern_ms, local.n_rows, local.nnz
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(per_rank)
    per_rank = per_rank.cpu().tolist()
    elapsed_ms = float(t.item())
    sec = elapsed_ms * 1e-3
    value = 2.0 * nnz_total * args.steps / sec / 1e9
    gbs = alg_bytes_total * args.steps / sec / 1e9
    eig = it.eigen_estimate()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, it.current_x(), eig)

    # ---- roofline of the dominant kernel on rank 0's shard
    alg_bytes_local = local.algorithmic_bytes()
    achieved = alg_bytes_local / (kern_ms * 1e-3) / 1e9 if kern_ms > 0 else None
    hot = spmv.hot_x_info(local.Aj)
    main_kernel = ("merge_tile_table_kernel" if hot["table_columns"] else
                   "merge_tile_hot_kernel" if hot["hot_columns"] else "merge_tile_reg_kernel") \
        if stats["chosen_kind"] == 0 else {1: "vector_kernel", 2: "light_kernel", 5: "stream_kernel"}.get(
            stats["chosen_kind"], "?")
    traffic, traffic_note = traffic_lookup(f"{args.workload}@{world}", main_kernel)

    # ---- parity, outside the timed region: one plain SpMV of this rank's row block against the
    # fp64 oracle on sampled rows; then the x replicas of all ranks bit for bit (what the fused
    # exchange -- peer stores or multicast -- wrote must be the same vector everywhere)
    x_now = it.current_x()
    y_chk = torch.full((local.n_rows,), float("nan"), dtype=local.Ax.dtype, device="cuda")
    spmv.spmv_ex(args.kind, local.Ap, local.Aj, local.Ax, x_now, y_chk, n_cols=n_cols)
    torch.cuda.synchronize()
    par = parity_leg(local, x_now, y_chk, seed=rank)
    del y_chk
    par_all = torch.tensor([[1.0 if par["ok"] else 0.0, par["max_err_over_scale"], par["rows_sampled"], 1.0]],
                           dtype=torch.float64, device="cuda").repeat(world, 1)
    if world > 1:
        ref = x_now.clone()
        dist.broadcast(ref, src=0)
        par_all[:, 3] = 1.0 if torch.equal(ref.view(torch.int32), x_now.view(torch.int32)) else 0.0
        del ref
        gathered = [torch.zeros_like(par_all[0]) for _ in range(world)]
        dist.all_gather(gathered, par_all[rank].contiguous())
        par_all = torch.stack(gathered)
    par_all = par_all.cpu().tolist()
    parity = {
        "ok": all(r[0] == 1.0 for r in par_all) and all(r[3] == 1.0 for r in par_all),
        "max_err_over_scale": max(r[1] for r in par_all), "tol": par["tol"],
        "rows_sampled": int(sum(r[2] for r in par_all)),
        "per_rank_ok": [r[0] == 1.0 for r in par_all],
        "x_replicas_bit_identical": all(r[3] == 1.0 for r in par_all) if world > 1 else None,
        "what": "one plain SpMV of every rank's row block vs " + par.get("oracle", "the fp64 oracle")
                + ("; then every rank's replica of x after the timed steps compared bit for bit with rank 0's"
                   if world > 1 else ""),
    }

    # ---- e2e: the host-buffer API, x H2D + kernel + y D2H every step, pinned host memory
    e2e = None

    def timed(fn):
        barrier()
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        td = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(td, op=dist.ReduceOp.MAX)
        return float(td.item())

    k, ns = args.e2e_steps, args.e2e_slots or (4 if world == 1 else 3)
    if k > 0 and world == 1:
        mat = CsrMatrix.from_device(local)
        xs = [torch.empty(n_cols, dtype=local.Ax.dtype, pin_memory=True) for _ in range(ns)]
        ys = [torch.empty(local.n_rows, dtype=local.Ax.dtype, pin_memory=True) for _ in range(ns)]
        xs[0].copy_(it.current_x().cpu())
        for t in xs[1:]:
            t.copy_(xs[0])
        xn, yn = [t.numpy() for t in xs], [t.numpy() for t in ys]
        for _ in range(2):
            mat.spmv(xn[0], yn[0], kind=args.kind)
        # one call at a time: upload, kernel, download, back to back
        dt_serial = timed(lambda: [mat.spmv(xn[0], yn[0], kind=args.kind) for _ in range(k)])
        # the pipelined call for a sequence of right-hand sides: `ns` slots in flight, so one
        # step's upload overlaps another step's kernel and a third's download
        mat.spmv_many([xn[i % ns] for i in range(ns)], [yn[i % ns] for i in range(ns)], kind=args.kind,
                      slots=ns)
        dt = timed(lambda: mat.spmv_many([xn[i % ns] for i in range(k)], [yn[i % ns] for i in range(k)],
                                         kind=args.kind, slots=ns))
        e2e = {"value": 2.0 * nnz_total * k / dt / 1e9, "unit": UNIT,
               "h2d_bytes_per_step": int(n_cols * xs[0].element_size()),
               "d2h_bytes_per_step": int(local.n_rows * ys[0].element_size()),
               "steps": k, "ms_per_step": dt / k * 1e3,
               "serial_value": 2.0 * nnz_total * k / dt_serial / 1e9,
               "serial_ms_per_step": dt_serial / k * 1e3,
               "api": "spmv_samples_b200.matrix.CsrMatrix.spmv_many (spmvb200_matrix_submit_host / "
                      "_wait): matrix resident (uploaded once, as reference main.cu:55-69); every "
                      "step uploads its x from pinned host memory, runs the SpMV and downloads y; "
                      f"{ns} steps in flight on {ns} streams.  serial_value: CsrMatrix.spmv, one step "
                      "at a time"}
        mat.close()
    elif k > 0:
        # row-sharded host-buffer call: every rank uploads its slice of x, the slices are
        # all-gathered over NVLink, every rank downloads its slice of y
        from spmv_samples_b200.dist import ShardedHostSpMV
        hs = ShardedHostSpMV(shard, n, kind=args.kind, slots=ns)
        rows_local = hs.io_end - hs.io_begin
        xs = [torch.empty(rows_local, dtype=local.Ax.dtype, pin_memory=True) for _ in range(ns)]
        ys = [torch.empty(rows_local, dtype=local.Ax.dtype, pin_memory=True) for _ in range(ns)]
        xs[0].copy_(it.current_x()[hs.io_begin:hs.io_end].cpu())
        for t in xs[1:]:
            t.copy_(xs[0])
        hs.spmv_many([xs[i % ns] for i in range(ns)], [ys[i % ns] for i in range(ns)])
        dt = timed(lambda: hs.spmv_many([xs[i % ns] for i in range(k)], [ys[i % ns] for i in range(k)]))
        e2e = {"value": 2.0 * nnz_total * k / dt / 1e9, "unit": UNIT,
               "h2d_bytes_per_step": int(n_cols * xs[0].element_size()),
               "d2h_bytes_per_step": int(n * ys[0].element_size()),
               "steps": k, "ms_per_step": dt / k * 1e3,
               "api": "spmv_samples_b200.dist.ShardedHostSpMV.spmv_many: matrix resident and "
                      "row-sharded (nnz-balanced); host I/O in even slices: every step each rank uploads "
                      "n/N values of x from pinned host memory, the slices are all-gathered over NVLink "
                      "(NCCL), the SpMV runs, the computed rows go to the ranks whose host slice they "
                      "belong to (one all-to-all, uneven splits) and each rank downloads n/N values of y; "
                      f"bytes are totals over the ranks; {ns} steps in flight"}
        hs.close()

    if e2e is not None:
        # what the host link takes for a step's copies alone (same pinned buffers, upload and
        # download at once on two streams, no kernel): e2e's ms_per_step cannot be far below it
        dx = torch.empty_like(xs[0], device="cuda")
        dy = torch.empty_like(ys[0], device="cuda")
        s_up, s_down = torch.cuda.Stream(), torch.cuda.Stream()

        def copies(rounds=6):
            for _ in range(rounds):
                with torch.cuda.stream(s_up):
                    dx.copy_(xs[0], non_blocking=True)
                with torch.cuda.stream(s_down):
                    ys[0].copy_(dy, non_blocking=True)
            s_up.synchronize()
            s_down.synchronize()
        copies(2)
        e2e["host_copies_alone_ms_per_step"] = timed(copies) / 6 * 1e3
        e2e["host_copies_note"] = ("a step's upload and download alone, both directions at once, from the same "
                                   "pinned buffers, no kernel (max over ranks): what this box's host link takes")
        del dx, dy

    exchange_used, exchange_note = it.exchange, getattr(it, "exchange_note", "")
    offset_bits = local.Ap.element_size() * 8
    value_dtype = "f32" if local.Ax.dtype == torch.float32 else "f64"
    it.close()
    configs = None
    if rank == 0 and world == 1 and not args.no_configs:
        del it, shard, local
        try:
            del gm
        except NameError:
            pass
        spmv.release_cache()
        torch.cuda.empty_cache()
        try:
            configs = configs_leg(peak)
        except Exception as e:
            configs = {"error": str(e)[:300]}
    if rank == 0:
        kind_names = {0: "merge", 1: "vector", 2: "light", 3: "auto", 4: "cusparse", 5: "stream"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": elapsed_ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": value_dtype,
            "data": "synthetic",
            "gbs": gbs, "roofline_frac_step": gbs / peak / world,
            "config": {
                "workload": workload_desc(args.workload, args.override), "seed": SEED,
                "rows": n, "nnz": nnz_total, "offset_bits": offset_bits,
                "algorithmic_bytes_per_spmv": alg_bytes_total,
                "step": "one power-iteration SpMV (x <- A x / ||A x||) over the whole matrix, "
                        "incl. x exchange and norm",
                "kind": args.kind, "selected_kernel": kind_names.get(stats["chosen_kind"]),
                "library_options": args.opts or None,
                "exchange": exchange_used, "exchange_note": exchange_note, "parallelism": f"row-sharded x{world} (merge-path nnz split, row weight {args.row_weight}"
                                + (f", re-split {args.rebalance}x from measured per-rank local step times)" if world > 1 and args.rebalance else ")"),
                "rebalance": rebalance_log,
                "l2": "inputs larger than L2 (no flush needed)" if alg_bytes_total > 4 * 126e6
                      else "inputs smaller than L2: steps run back to back, L2-warm",
                "generation_s": t_gen, "eigen_estimate": eig,
                "row_stats": {k: stats[k] for k in ("max_row_len", "mean_row_len", "std_row_len", "empty_rows")},
                "hot_x": dict(hot, note="merge-path kernel gathers the most frequent columns from a dense "
                              "copy refilled from x every step (csrc/hotx.cu); plan built once, outside the timed region"),
                "per_rank": {"kernel_ms": [round(r[0], 4) for r in per_rank],
                             "rows": [int(r[1]) for r in per_rank], "nnz": [int(r[2]) for r in per_rank]},
            },
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                         "traffic_note": traffic_note,
                         "peak_source": peak_src, "kernel_ms": kern_ms,
                         "kernel": f"{main_kernel} ({kind_names.get(stats['chosen_kind'])} main kernel), rank 0 shard",
                         "algorithmic_bytes_per_launch": alg_bytes_local,
                         "kernel_share_of_step": kern_ms / (elapsed_ms / args.steps),
                         "non_kernel_ms": elapsed_ms / args.steps - kern_ms,
                         "frac_of_datasheet_8000": (achieved / 8000.0) if achieved else None},
            "cpu_baseline": cpu_info,
            "parity": parity,
            "configs": configs,
            "e2e": e2e,
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def C_double():
    import ctypes
    return ctypes.c_double(0.0)


def C_int64():
    import ctypes
    return ctypes.c_int64(0)


def main():
    args = parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        return reference_arm(args, rank, world)
    from spmv_samples_b200.dist import init_distributed
    rank, world, local_rank = init_distributed()
    if world != args.gpus and rank == 0:
        print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; using {world}", file=sys.stderr)
    return own_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    sys.exit(main())
