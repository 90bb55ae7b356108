// main.cu -- the bench driver: same command line and output sections as reference/main.cu
// ("Dataset", "Compute delta", "Time cost"), same flow (load .mtx -> CSR -> device copies ->
// host check -> per-kind correctness -> per-kind timing loop of TEST_TIMES calls), rebuilt on
// the C-ABI library:
//
//   ./bin/spmv <filename.mtx | synthetic:c1..c5[:size]> <SpMV_kind_string>... [options]
//
// What changes (BASELINE.json north_star, SURVEY.md 2.1 row 1):
//   * timing is cudaEvent time on the SpMV stream (include/timer.hpp), reported in
//     microseconds with the right label (the reference prints microseconds as "ms"), plus
//     GFLOP/s = 2 nnz / t, effective GB/s on the algorithmic byte count, and the fraction of the
//     HBM roofline (measured copy bandwidth and datasheet, both labelled);
//   * the self-check has a tolerance and an exit code: |y - y_ref| <= tol * sum_j |a_ij x_j|
//     per row against an fp64 host reference (tol 1e-5 fp32, 1e-13 fp64);
//   * synthetic matrices of the five configurations, generated on the device;
//   * the host CSR loop is timed too (one thread, like the reference's), as a reported baseline.
// Options: --iters N (default 2000, reference/main.cu:19)   --x ones|random (default ones,
//   reference/main.cu:41)   --flush (evict L2 between timed calls)   --peak GBps
//   --dynamic-pattern: the timing loop does not declare the matrix unchanged between calls (the
//   default does, through option "assume_static_pattern": partition and hot-x plan are reused)
//   --power K [--gpus N]: K power-iteration steps, the matrix row-sharded over N GPUs of the box
//   (one process, peer access; csrc/multi.cu) -- the multi-GPU configuration without Python
//   --cg RTOL [--jacobi]: for a square matrix, b = A*1 and x0 = 0, then one conjugate-gradient solve
//   (Jacobi-preconditioned with --jacobi) per kind through spmvb200_cg; exits non-zero if one does
//   not converge
//   --bicgstab RTOL [--jacobi]: the same with one BiCGSTAB solve per kind (spmvb200_bicgstab), for a
//   square matrix that need not be symmetric
//   --gmres RTOL [--restart M] [--jacobi]: the same with one restarted GMRES(M) solve per kind
//   (spmvb200_gmres, M = 20 by default, at most 64), for a square matrix that need not be symmetric
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <filesystem>
#include <functional>
#include <iostream>
#include <numeric>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "load.hpp"
#include "spmv.h"

using namespace std;

using index_t = int;

constexpr int TEST_TIMES = 2000;

struct Options {
    string input;
    vector<string> kinds;
    int iters = TEST_TIMES;
    bool random_x = false;
    bool flush = false;
    bool static_pattern = true;  // --dynamic-pattern: do not vouch for an unchanged matrix in the timing loop
    double peak_gbs = 6452.2;  // fallback: this pool's measured copy bandwidth; MEASURED_PEAKS.json beside
                               // the working directory, or --peak, overrides it
    double datasheet_gbs = 8000.0;
    uint64_t seed = 0x5EEDB200ull;
    int gpus = 1;    // --gpus N: the row-sharded power iteration over N GPUs of this box
    int power = 0;   // --power K: K power-iteration steps x <- A x / ||A x|| (BASELINE.json configs[4])
    double cg_rtol = 0;      // --cg RTOL: one CG solve of A x = A*1 per kind
    double bicgstab_rtol = 0;  // --bicgstab RTOL: one BiCGSTAB solve of A x = A*1 per kind
    double gmres_rtol = 0;     // --gmres RTOL: one GMRES solve of A x = A*1 per kind
    int gmres_restart = 20;    // --restart M: GMRES cycle length
    bool cg_jacobi = false;  // --jacobi: with M = diag(A) (every solver)
};

template <typename T>
static T *device_alloc(size_t n) {
    T *p = nullptr;
    checkCudaErr(cudaMalloc((void **)&p, std::max<size_t>(n, 1) * sizeof(T)));
    return p;
}

// the SpMV kind behind a label of the kind table (include/spmv.h), or -1
static int kind_id(const string &k) {
    if (k == "merge" || k == "cub_merge" || k == "merge_genl") return SPMVB200_KIND_MERGE;
    if (k == "vector" || k == "cusp" || k == "cusp1" || k == "cusp2") return SPMVB200_KIND_VECTOR;
    if (k == "light" || k == "light_vec" || k == "light_warp") return SPMVB200_KIND_LIGHT;
    if (k == "stream") return SPMVB200_KIND_STREAM;
    if (k == "auto") return SPMVB200_KIND_AUTO;
    if (k == "cusparse") return SPMVB200_KIND_CUSPARSE;
    return -1;
}

using KrylovSolve = std::function<int(const spmvb200_cg_args_t *, spmvb200_cg_result_t *)>;

// --cg / --bicgstab / --gmres: b = A*1, x0 = 0, one solve per kind by `solve` (spmvb200_cg,
// spmvb200_bicgstab or spmvb200_gmres); returns the number of kinds that did not converge
template <typename offset_t, typename value_t>
static int run_krylov(const Options &opt, const KrylovSolve &solve, const char *title, double rtol, index_t n, offset_t nnz,
                      offset_t *dAp, index_t *dAj, value_t *dAx) {
    const size_t vb = sizeof(value_t);
    vector<value_t> ones((size_t)n, value_t(1)), hx((size_t)n);
    value_t *d1 = device_alloc<value_t>((size_t)n), *dB = device_alloc<value_t>((size_t)n);
    value_t *dX = device_alloc<value_t>((size_t)n);
    checkCudaErr(cudaMemcpy(d1, ones.data(), (size_t)n * vb, cudaMemcpyHostToDevice));
    spmvb200_args_t s;
    memset(&s, 0, sizeof(s));
    s.kind = SPMVB200_KIND_MERGE;
    s.offset_bits = sizeof(offset_t) * 8;
    s.value_bits = vb * 8;
    s.n_rows = s.n_cols = n;
    s.nnz = (int64_t)nnz;
    s.Ap = dAp;
    s.Aj = dAj;
    s.Ax = dAx;
    s.x = d1;
    s.y = dB;
    checkSpmvStatus(spmvb200_spmv(&s));
    checkCudaErr(cudaDeviceSynchronize());
    cudaEvent_t e0, e1;
    checkCudaErr(cudaEventCreate(&e0));
    checkCudaErr(cudaEventCreate(&e1));
    printf("%s (b = A*1, x0 = 0, rtol %.1e%s, max %d iterations):\n", title, rtol,
           opt.cg_jacobi ? ", Jacobi preconditioner" : "", n);
    int failures = 0;
    for (const auto &kind : opt.kinds) {
        const int id = kind_id(kind);
        if (id < 0) {
            printf("[%-12s] no such kind\n", kind.data());
            ++failures;
            continue;
        }
        checkCudaErr(cudaMemset(dX, 0, (size_t)n * vb));
        spmvb200_cg_args_t a;
        memset(&a, 0, sizeof(a));
        a.kind = id;
        a.offset_bits = sizeof(offset_t) * 8;
        a.value_bits = vb * 8;
        a.flags = opt.cg_jacobi ? SPMVB200_CG_JACOBI : 0;
        a.n = n;
        a.nnz = (int64_t)nnz;
        a.Ap = dAp;
        a.Aj = dAj;
        a.Ax = dAx;
        a.b = dB;
        a.x = dX;
        a.rtol = rtol;
        a.max_iter = n;
        spmvb200_cg_result_t r;
        checkCudaErr(cudaEventRecord(e0, nullptr));
        checkSpmvStatus(solve(&a, &r));  // synchronises
        checkCudaErr(cudaEventRecord(e1, nullptr));
        checkCudaErr(cudaEventSynchronize(e1));
        float ms = 0.f;
        checkCudaErr(cudaEventElapsedTime(&ms, e0, e1));
        checkCudaErr(cudaMemcpy(hx.data(), dX, (size_t)n * vb, cudaMemcpyDeviceToHost));
        double err = 0.0;
        for (index_t i = 0; i < n; ++i) err = std::max(err, std::abs((double)hx[(size_t)i] - 1.0));
        failures += !r.converged;
        printf("[%-12s] %lld iterations  |b-Ax|/|b| = %.3e  max|x-1| = %.3e  %.3f ms  %.4f ms/iteration  %s\n",
               kind.data(), (long long)r.iterations, r.b_norm > 0 ? r.residual_norm / r.b_norm : r.residual_norm, err,
               ms, r.iterations ? ms / r.iterations : 0.0,
               r.converged ? "CONVERGED" : r.breakdown ? "BREAKDOWN" : "NOT CONVERGED");
    }
    checkCudaErr(cudaEventDestroy(e0));
    checkCudaErr(cudaEventDestroy(e1));
    checkCudaErr(cudaFree(d1));
    checkCudaErr(cudaFree(dB));
    checkCudaErr(cudaFree(dX));
    return failures;
}

template <typename offset_t, typename value_t>
static int run(const Options &opt, const string &name, index_t n_rows, index_t n_cols, offset_t nnz,
               offset_t *dA_csrOffsets, index_t *dA_columns, value_t *dA_values,
               const vector<offset_t> &hAp, const vector<index_t> &hAj, const vector<value_t> &hAx,
               index_t check_rows) {
    cout << "Dataset: " << name << endl
         << "\tn_rows: " << n_rows << "  n_cols: " << n_cols << "  nnz: " << nnz << endl;

    // x: all ones like the reference driver, or seeded U(-1,1) (catches wrong column indices)
    vector<value_t> vec_x((size_t)n_cols, value_t(1));
    value_t *dX = device_alloc<value_t>((size_t)n_cols);
    value_t *dY = device_alloc<value_t>((size_t)n_rows);
    if (opt.random_x) {
        checkSpmvStatus(spmvb200_gen_uniform_pm1(sizeof(value_t) * 8, opt.seed, 2, 0, n_cols, dX, nullptr));
        checkCudaErr(cudaMemcpy(vec_x.data(), dX, (size_t)n_cols * sizeof(value_t), cudaMemcpyDeviceToHost));
    } else {
        checkCudaErr(cudaMemcpy(dX, vec_x.data(), (size_t)n_cols * sizeof(value_t), cudaMemcpyHostToDevice));
    }
    vector<value_t> vec_y((size_t)n_rows, value_t(0));

    //--------------------------------------------------------------------------
    // host check (fp64), timed as the single-thread CPU baseline
    vector<double> correct_y, scale;
    auto t0 = chrono::steady_clock::now();
    SpMV_host_check(check_rows, hAp.data(), hAj.data(), hAx.data(), vec_x.data(), correct_y, scale);
    const double cpu_s = chrono::duration<double>(chrono::steady_clock::now() - t0).count();
    const double checked_nnz = (double)hAp[(size_t)check_rows];
    const double tol = sizeof(value_t) == 4 ? 1e-5 : 1e-13;

    int failures = 0;
    printf("Compute delta:\n");
    for (const auto &kind : opt.kinds) {
        checkCudaErr(cudaMemset(dY, 0xff, (size_t)n_rows * sizeof(value_t)));  // NaN pattern
        SpMV(kind, n_rows, n_cols, nnz, dA_csrOffsets, dA_columns, dA_values, dX, dY);
        checkCudaErr(cudaDeviceSynchronize());
        checkCudaErr(cudaMemcpy(vec_y.data(), dY, (size_t)n_rows * sizeof(value_t), cudaMemcpyDeviceToHost));
        double delta = 0., worst = 0.;
        size_t bad = 0;
        for (index_t i = 0; i < check_rows; ++i) {
            const double d = std::abs(correct_y[(size_t)i] - (double)vec_y[(size_t)i]);
            delta += d;
            if (!(d <= tol * scale[(size_t)i])) ++bad;
            if (scale[(size_t)i] > 0) worst = std::max(worst, d / scale[(size_t)i]);
        }
        failures += bad != 0;
        printf("[%-12s] sum: %12lf  avg: %12lf  worst |dy|/sum|a x|: %.3e  %s (tol %.0e, %d rows checked)\n",
               kind.data(), delta, delta / std::max<index_t>(check_rows, 1), worst,
               bad ? "FAIL" : "PASS", tol, check_rows);
    }
    printf("\n");

    //--------------------------------------------------------------------------
    // time cost
    const double bytes = (double)nnz * (sizeof(index_t) + sizeof(value_t)) +
                         ((double)n_rows + 1) * sizeof(offset_t) + (double)n_cols * sizeof(value_t) +
                         (double)n_rows * sizeof(value_t);
    const double flops = 2.0 * (double)nnz;
    char *flush_buf = nullptr;
    const size_t flush_bytes = 512ull << 20;
    if (opt.flush) checkCudaErr(cudaMalloc((void **)&flush_buf, flush_bytes));
    // Two ways of timing, both in device time.  With --flush every call is bracketed by its own
    // event pair and the host waits for it (the flush in between is not counted).  Without it the
    // calls are queued back to back, as in reference/main.cu:104-110, inside ONE event pair and
    // the host synchronises once after the loop: no launch latency or idle gap between calls is
    // counted as kernel time, and none is hidden either.
    // The timing loop calls every kind on one unchanged matrix, which the SpMV(kind_str, ...)
    // signature cannot say: the driver says it through a library option, so that the calls may
    // reuse the merge-path partition and the hot-x plan (spmv_b200.h, SPMVB200_FLAG_STATIC_PATTERN).
    // The check above ran without it.
    checkSpmvStatus(spmvb200_set_option("assume_static_pattern", opt.static_pattern ? 1 : 0));
    printf("Time cost (%d calls%s%s; %.0f algorithmic bytes, %.0f flops per call):\n", opt.iters,
           opt.flush ? ", L2 flushed before each, timed one by one" : ", queued back to back, timed as one interval",
           opt.static_pattern ? ", matrix declared unchanged between calls" : "", bytes, flops);
    cudaEvent_t loop_begin, loop_end;
    checkCudaErr(cudaEventCreate(&loop_begin));
    checkCudaErr(cudaEventCreate(&loop_end));
    for (const auto &kind : opt.kinds) {
        for (int i = 0; i < 3; ++i)  // warm-up (scratch allocation, statistics cache)
            SpMV(kind, n_rows, n_cols, nnz, dA_csrOffsets, dA_columns, dA_values, dX, dY);
        double total_time = 0, kernel_time = 0;
        if (opt.flush) {
            for (int i = 0; i < opt.iters; ++i) {
                checkCudaErr(cudaMemsetAsync(flush_buf, i & 0xff, flush_bytes, SpmvStream::get()));
                SpMV(kind, n_rows, n_cols, nnz, dA_csrOffsets, dA_columns, dA_values, dX, dY);
                total_time += Timer::total_cost_us();
                kernel_time += Timer::kernel_cost_us();
            }
        } else {
            checkCudaErr(cudaEventRecord(loop_begin, SpmvStream::get()));
            for (int i = 0; i < opt.iters; ++i)
                SpMV(kind, n_rows, n_cols, nnz, dA_csrOffsets, dA_columns, dA_values, dX, dY);
            checkCudaErr(cudaEventRecord(loop_end, SpmvStream::get()));
            checkCudaErr(cudaEventSynchronize(loop_end));
            float ms = 0.f;
            checkCudaErr(cudaEventElapsedTime(&ms, loop_begin, loop_end));
            total_time = kernel_time = (double)ms * 1e3;
        }
        const double t_us = kernel_time / opt.iters;
        const double gbs = bytes / (t_us * 1e-6) / 1e9;
        printf("[%-12s] total: %12lf us  kernel: %12lf us  %9.1f GFLOP/s  %8.1f GB/s  "
               "%5.1f%% of measured %.0f GB/s  %5.1f%% of datasheet %.0f GB/s\n",
               kind.data(), total_time / opt.iters, t_us, flops / (t_us * 1e-6) / 1e9, gbs,
               100.0 * gbs / opt.peak_gbs, opt.peak_gbs, 100.0 * gbs / opt.datasheet_gbs, opt.datasheet_gbs);
    }
    printf("[%-12s] %.3f ms for %.0f nonzeros on 1 host thread: %.2f GFLOP/s (reported baseline)\n",
           "cpu fp64", cpu_s * 1e3, checked_nnz, 2.0 * checked_nnz / cpu_s / 1e9);

    checkSpmvStatus(spmvb200_set_option("assume_static_pattern", 0));
    checkCudaErr(cudaEventDestroy(loop_begin));
    checkCudaErr(cudaEventDestroy(loop_end));
    //--------------------------------------------------------------------------
    // power iteration, row-sharded over --gpus GPUs from this one process (csrc/multi.cu): the
    // matrix goes from this device to the others by peer copies; the iteration itself never
    // returns to the host
    if (opt.power > 0 && n_rows == n_cols) {
        spmvb200_power_t *pw = nullptr;
        checkSpmvStatus(spmvb200_power_create_from_device(opt.gpus, nullptr, sizeof(offset_t) * 8, sizeof(value_t) * 8,
                                                          n_rows, (int64_t)nnz, dA_csrOffsets, dA_columns, dA_values,
                                                          SPMVB200_KIND_AUTO, &pw));
        double ms = 0, norm = 0;
        checkSpmvStatus(spmvb200_power_run(pw, 5, &ms));   // warm-up: scratch, statistics, hot-x plan
        checkSpmvStatus(spmvb200_power_reset(pw));
        checkSpmvStatus(spmvb200_power_run(pw, opt.power, &ms));
        vector<int64_t> rb((size_t)opt.gpus + 1);
        checkSpmvStatus(spmvb200_power_get(pw, nullptr, &norm, rb.data()));
        printf("Power iteration (%d steps, %d GPU%s, kind auto%s):\n", opt.power, opt.gpus, opt.gpus > 1 ? "s" : "",
               opt.gpus < 2 ? "" : spmvb200_power_exchange(pw) ? ", rows exchanged by NVLink multicast stores" : ", rows exchanged by peer stores");
        printf("[%-12s] %12lf ms/step  %9.1f GFLOP/s  %8.1f GB/s  %5.1f%% of measured %.0f GB/s x %d  ||A x|| = %.9g\n",
               "power", ms, flops / (ms * 1e-3) / 1e9, bytes / (ms * 1e-3) / 1e9,
               100.0 * bytes / (ms * 1e-3) / 1e9 / (opt.peak_gbs * opt.gpus), opt.peak_gbs, opt.gpus, norm);
        printf("[%-12s] rows per GPU:", "split");
        for (int g = 0; g < opt.gpus; ++g) printf(" %lld", (long long)(rb[(size_t)g + 1] - rb[(size_t)g]));
        printf("\n");
        spmvb200_power_destroy(pw);
    }

    const struct {
        double rtol;
        KrylovSolve solve;
        const char *title;
    } solves[] = {{opt.cg_rtol, spmvb200_cg, "Conjugate gradients"},
                  {opt.bicgstab_rtol, spmvb200_bicgstab, "BiCGSTAB"},
                  {opt.gmres_rtol,
                   [&opt](const spmvb200_cg_args_t *a, spmvb200_cg_result_t *r) {
                       return spmvb200_gmres(a, opt.gmres_restart, r);
                   },
                   "GMRES"}};
    for (const auto &sv : solves) {
        if (sv.rtol <= 0) continue;
        if (n_rows == n_cols) {
            failures += run_krylov<offset_t, value_t>(opt, sv.solve, sv.title, sv.rtol, n_rows, nnz, dA_csrOffsets,
                                                      dA_columns, dA_values);
        } else {
            printf("%s: the matrix is not square\n", sv.title);
            ++failures;
        }
    }

    if (flush_buf) checkCudaErr(cudaFree(flush_buf));
    checkCudaErr(cudaFree(dX));
    checkCudaErr(cudaFree(dY));
    return failures;
}

// .mtx file through the host loader, types as in reference/main.cu:15-17
static int run_file(const Options &opt) {
    using offset_t = int;
    using value_t = float;
    csr_t<index_t, offset_t, value_t> csr = ToCsr(LoadCoo<index_t, offset_t, value_t>(opt.input));
    const index_t n_rows = csr.number_of_rows, n_cols = csr.number_of_columns;
    const offset_t nnz = csr.number_of_nonzeros;
    offset_t *dAp = device_alloc<offset_t>((size_t)n_rows + 1);
    index_t *dAj = device_alloc<index_t>((size_t)nnz);
    value_t *dAx = device_alloc<value_t>((size_t)nnz);
    checkCudaErr(cudaMemcpy(dAp, csr.row_offsets.data(), ((size_t)n_rows + 1) * sizeof(offset_t), cudaMemcpyHostToDevice));
    checkCudaErr(cudaMemcpy(dAj, csr.column_indices.data(), (size_t)nnz * sizeof(index_t), cudaMemcpyHostToDevice));
    checkCudaErr(cudaMemcpy(dAx, csr.nonzero_values.data(), (size_t)nnz * sizeof(value_t), cudaMemcpyHostToDevice));
    const int rc = run<offset_t, value_t>(opt, filesystem::path(opt.input).filename().string(), n_rows, n_cols, nnz,
                                          dAp, dAj, dAx, csr.row_offsets, csr.column_indices,
                                          csr.nonzero_values, n_rows);
    checkCudaErr(cudaFree(dAp));
    checkCudaErr(cudaFree(dAj));
    checkCudaErr(cudaFree(dAx));
    return rc;
}

// synthetic:<config>[:size] generated on the device, copied back for the host check
template <typename offset_t, typename value_t>
static int run_synthetic(const Options &opt, const string &cfg, long size) {
    const int ob = sizeof(offset_t) * 8, vb = sizeof(value_t) * 8;
    index_t n_rows = 0, n_cols = 0;
    int64_t nnz = 0;
    offset_t *dAp = nullptr;
    index_t *dAj = nullptr;
    value_t *dAx = nullptr;
    if (cfg == "c1") {
        const int g = size > 0 ? (int)size : 1024;
        n_rows = n_cols = g * g;
        nnz = 5ll * n_rows - 4ll * g;
        dAp = device_alloc<offset_t>((size_t)n_rows + 1);
        dAj = device_alloc<index_t>((size_t)nnz);
        dAx = device_alloc<value_t>((size_t)nnz);
        checkSpmvStatus(spmvb200_gen_lap2d(ob, vb, g, dAp, dAj, dAx, nullptr));
    } else if (cfg == "c2" || cfg == "c4") {
        const int K = cfg == "c2" ? 16 : 2048;
        n_rows = n_cols = size > 0 ? (index_t)size : (cfg == "c2" ? 4 << 20 : 65536);
        nnz = (int64_t)n_rows * K;
        dAp = device_alloc<offset_t>((size_t)n_rows + 1);
        dAj = device_alloc<index_t>((size_t)nnz);
        dAx = device_alloc<value_t>((size_t)nnz);
        checkSpmvStatus(spmvb200_gen_uniform_rows(ob, vb, n_rows, n_cols, K, opt.seed, dAp, dAj, dAx, nullptr));
    } else {  // c3, c5: R-MAT
        const int scale = size > 0 ? (int)size : (cfg == "c3" ? 24 : 27);
        n_rows = n_cols = 1 << scale;
        nnz = 16ll * n_rows;
        index_t *rows = device_alloc<index_t>((size_t)nnz), *cols = device_alloc<index_t>((size_t)nnz);
        dAp = device_alloc<offset_t>((size_t)n_rows + 1);
        dAj = device_alloc<index_t>((size_t)nnz);
        dAx = device_alloc<value_t>((size_t)nnz);
        checkSpmvStatus(spmvb200_gen_rmat_edges(scale, opt.seed, 0, nnz, rows, cols, nullptr));
        checkSpmvStatus(spmvb200_coo_to_csr(ob, vb, n_rows, nnz, rows, cols, nullptr, dAp, dAj, nullptr, nullptr));
        checkCudaErr(cudaFree(rows));
        checkCudaErr(cudaFree(cols));
        checkSpmvStatus(spmvb200_gen_uniform_pm1(vb, opt.seed, 1, 0, nnz, dAx, nullptr));
    }
    checkCudaErr(cudaDeviceSynchronize());
    // host copy: everything up to 2^28 nonzeros, else a prefix of rows holding about that many
    vector<offset_t> hAp((size_t)n_rows + 1);
    checkCudaErr(cudaMemcpy(hAp.data(), dAp, hAp.size() * sizeof(offset_t), cudaMemcpyDeviceToHost));
    index_t check_rows = n_rows;
    const int64_t cap = 1ll << 28;
    if (nnz > cap) check_rows = (index_t)(std::upper_bound(hAp.begin(), hAp.end(), (offset_t)cap) - hAp.begin() - 1);
    const size_t h_nnz = (size_t)hAp[(size_t)check_rows];
    vector<index_t> hAj(h_nnz);
    vector<value_t> hAx(h_nnz);
    checkCudaErr(cudaMemcpy(hAj.data(), dAj, h_nnz * sizeof(index_t), cudaMemcpyDeviceToHost));
    checkCudaErr(cudaMemcpy(hAx.data(), dAx, h_nnz * sizeof(value_t), cudaMemcpyDeviceToHost));
    const int rc = run<offset_t, value_t>(opt, "synthetic:" + cfg, n_rows, n_cols, (offset_t)nnz, dAp, dAj, dAx,
                                          hAp, hAj, hAx, check_rows);
    checkCudaErr(cudaFree(dAp));
    checkCudaErr(cudaFree(dAj));
    checkCudaErr(cudaFree(dAx));
    return rc;
}

int main(int argc, char **argv) {
    if (argc < 3) {
        cerr << "usage: ./bin/<program-name>  <filename.mtx | synthetic:c1..c5[:size]>  <SpMV_kind_string>..."
                "  [--iters N] [--x ones|random] [--flush] [--dynamic-pattern] [--peak GB/s] [--power K [--gpus N]] [--cg RTOL] [--bicgstab RTOL] [--gmres RTOL [--restart M]] [--jacobi]"
             << endl;
        exit(1);
    }
    Options opt;
    opt.input = argv[1];
    for (int i = 2; i < argc; ++i) {
        const string a = argv[i];
        if (a == "--iters" && i + 1 < argc) opt.iters = atoi(argv[++i]);
        else if (a == "--x" && i + 1 < argc) opt.random_x = string(argv[++i]) == "random";
        else if (a == "--flush") opt.flush = true;
        else if (a == "--dynamic-pattern") opt.static_pattern = false;
        else if (a == "--peak" && i + 1 < argc) opt.peak_gbs = atof(argv[++i]);
        else if (a == "--gpus" && i + 1 < argc) opt.gpus = atoi(argv[++i]);
        else if (a == "--power" && i + 1 < argc) opt.power = atoi(argv[++i]);
        else if (a == "--cg" && i + 1 < argc) opt.cg_rtol = atof(argv[++i]);
        else if (a == "--bicgstab" && i + 1 < argc) opt.bicgstab_rtol = atof(argv[++i]);
        else if (a == "--gmres" && i + 1 < argc) opt.gmres_rtol = atof(argv[++i]);
        else if (a == "--restart" && i + 1 < argc) opt.gmres_restart = atoi(argv[++i]);
        else if (a == "--jacobi") opt.cg_jacobi = true;
        else opt.kinds.push_back(a);
    }
    if (opt.kinds.empty() || opt.iters < 1) {
        cerr << "no SpMV kind given" << endl;
        exit(1);
    }

    checkCudaErr(cudaSetDevice(USED_DEVICE));
    {   // the roofline denominator: MEASURED_PEAKS.json ("hbm_gbs": ...) if it can be found
        bool peak_given = false;
        for (int i = 2; i < argc; ++i) peak_given = peak_given || string(argv[i]) == "--peak";
        if (!peak_given) {
            for (const char *path : {"MEASURED_PEAKS.json", "../MEASURED_PEAKS.json"}) {
                if (FILE *f = fopen(path, "r")) {
                    char buf[4096];
                    const size_t n = fread(buf, 1, sizeof(buf) - 1, f);
                    fclose(f);
                    buf[n] = 0;
                    if (const char *k = strstr(buf, "\"hbm_gbs\"")) {
                        if (const char *c = strchr(k, ':')) {
                            const double v = atof(c + 1);
                            if (v > 0) opt.peak_gbs = v;
                        }
                    }
                    break;
                }
            }
        }
    }

    int failures = 0;
    if (opt.input.rfind("synthetic:", 0) == 0) {
        string cfg = opt.input.substr(10);
        long size = 0;
        const size_t colon = cfg.find(':');
        if (colon != string::npos) {
            size = atol(cfg.substr(colon + 1).c_str());
            cfg = cfg.substr(0, colon);
        }
        if (cfg == "c1" || cfg == "c2" || cfg == "c3") failures = run_synthetic<int, float>(opt, cfg, size);
        else if (cfg == "c4") failures = run_synthetic<int, double>(opt, cfg, size);
        else if (cfg == "c5") failures = run_synthetic<int64_t, float>(opt, cfg, size);
        else {
            cerr << "unknown synthetic configuration \"" << cfg << "\" (c1..c5)" << endl;
            exit(1);
        }
    } else {
        failures = run_file(opt);
    }
    return failures ? EXIT_FAILURE : EXIT_SUCCESS;
}
