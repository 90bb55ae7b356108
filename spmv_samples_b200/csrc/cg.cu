// cg.cu -- conjugate gradients on a symmetric positive definite CSR matrix, optionally with the
// Jacobi preconditioner M = diag(A), entirely on the device (spmvb200_cg).
//
// One iteration is the caller's SpMV kind (q = A p, through spmvb200_spmv with
// SPMVB200_FLAG_STATIC_PATTERN) followed by three streaming kernels:
//   cg_pq_kernel         p.q                          -> alpha = rho / p.q   (breakdown if p.q <= 0)
//   cg_update_kernel     x += alpha p, r -= alpha q, z = dinv r (Jacobi); r.z, r.r
//                                                     -> beta = rho' / rho, converged, iteration += 1
//   cg_direction_kernel  p = z + beta p
// Every dot product accumulates in double in a fixed order (grid_sum, krylov.cuh).  The scalars
// live in a small device state block, so the host never reads them inside the loop: it enqueues
// iterations in batches of 1, 2, 4, ... kKrylovMaxBatch and reads the flags once per batch.  Every CG kernel returns at once when `converged` or `breakdown` is set, so x and the
// iteration count are those of the iteration where the criterion first held, whatever the batch
// boundaries (the SpMVs left in a batch still run; they only rewrite q).
#include <algorithm>
#include <cmath>
#include <cstring>

#include "krylov.cuh"

namespace spmvb200 {
namespace {

struct CgState {
    double rho;    // r.z of the current residual
    double alpha;  // rho / p.q
    double beta;   // rho_new / rho
    double rr;     // ||r||^2 of the recursive residual
    double bb;     // ||b||^2
    double tol;    // rtol * ||b||
    double res2;   // ||b - A x||^2 of the returned x, in fp64
    unsigned long long iterations;
    int converged;
    int breakdown;
    int bad_diag;             // Jacobi: a row without a (non-zero) diagonal entry
    unsigned int counter;     // blocks finished in the running reduction; the last one resets it
};

__device__ __forceinline__ bool cg_stopped(const CgState *st) { return (st->converged | st->breakdown) != 0; }

// r = b - q (q = A x0), z = dinv r, p = z; rho = r.z, ||r||^2, ||b||^2
template <typename ValT, bool kJacobi>
__global__ void __launch_bounds__(kKrylovBlock)
cg_init_kernel(int64_t n, const ValT *__restrict__ b, const ValT *__restrict__ q, const ValT *__restrict__ dinv,
               ValT *__restrict__ r, ValT *__restrict__ z, ValT *__restrict__ p, double rtol, CgState *st,
               double *__restrict__ partial) {
    double acc[3] = {0.0, 0.0, 0.0};  // r.z, r.r, b.b
    for (int64_t i = first_index(); i < n; i += grid_stride()) {
        const ValT bi = b[i];
        const ValT ri = bi - q[i];
        r[i] = ri;
        ValT zi = ri;
        if (kJacobi) {
            zi = dinv[i] * ri;
            z[i] = zi;
        }
        p[i] = zi;
        acc[0] += (double)ri * (double)zi;
        acc[1] += (double)ri * (double)ri;
        acc[2] += (double)bi * (double)bi;
    }
    if (!grid_sum<3>(acc, partial, &st->counter)) return;
    if (threadIdx.x == 0) {
        st->rho = acc[0];
        st->rr = acc[1];
        st->bb = acc[2];
        st->tol = rtol * sqrt(acc[2]);
        st->iterations = 0;
        if (acc[2] == 0.0 || sqrt(acc[1]) <= st->tol) st->converged = 1;
        else if (!(acc[0] > 0.0) || !isfinite(acc[0])) st->breakdown = 1;
    }
}

// p.q -> alpha
template <typename ValT>
__global__ void __launch_bounds__(kKrylovBlock)
cg_pq_kernel(int64_t n, const ValT *__restrict__ p, const ValT *__restrict__ q, CgState *st,
             double *__restrict__ partial) {
    if (cg_stopped(st)) return;
    double acc[1] = {0.0};
    for (int64_t i = first_index(); i < n; i += grid_stride()) acc[0] += (double)p[i] * (double)q[i];
    if (!grid_sum<1>(acc, partial, &st->counter)) return;
    if (threadIdx.x == 0) {
        const double pq = acc[0];
        if (!(pq > 0.0) || !isfinite(pq)) st->breakdown = 1;
        else st->alpha = st->rho / pq;
    }
}

// x += alpha p, r -= alpha q, z = dinv r; r.z and r.r -> converged / beta, one more iteration
template <typename ValT, bool kJacobi>
__global__ void __launch_bounds__(kKrylovBlock)
cg_update_kernel(int64_t n, const ValT *__restrict__ p, const ValT *__restrict__ q, const ValT *__restrict__ dinv,
                 ValT *__restrict__ x, ValT *__restrict__ r, ValT *__restrict__ z, CgState *st,
                 double *__restrict__ partial) {
    if (cg_stopped(st)) return;
    const ValT a = (ValT)st->alpha;
    constexpr int N = kJacobi ? 2 : 1;
    double acc[N];  // r.r (, r.z)
#pragma unroll
    for (int j = 0; j < N; ++j) acc[j] = 0.0;
    for (int64_t i = first_index(); i < n; i += grid_stride()) {
        x[i] += a * p[i];
        const ValT ri = r[i] - a * q[i];
        r[i] = ri;
        acc[0] += (double)ri * (double)ri;
        if (kJacobi) {
            const ValT zi = dinv[i] * ri;
            z[i] = zi;
            acc[N - 1] += (double)ri * (double)zi;
        }
    }
    if (!grid_sum<N>(acc, partial, &st->counter)) return;
    if (threadIdx.x == 0) {
        const double rr = acc[0], rz = acc[N - 1];
        st->rr = rr;
        st->iterations += 1;
        if (sqrt(rr) <= st->tol) {
            st->converged = 1;
        } else if (!(rz > 0.0) || !isfinite(rz)) {
            st->breakdown = 1;
        } else {
            st->beta = rz / st->rho;
            st->rho = rz;
        }
    }
}

// p = z + beta p  (z = r without a preconditioner)
template <typename ValT>
__global__ void __launch_bounds__(kKrylovBlock)
cg_direction_kernel(int64_t n, const ValT *__restrict__ z, ValT *__restrict__ p, const CgState *st) {
    if (cg_stopped(st)) return;
    const ValT bt = (ValT)st->beta;
    for (int64_t i = first_index(); i < n; i += grid_stride()) p[i] = z[i] + bt * p[i];
}

template <typename OffT, typename ValT, bool kJacobi>
int cg_run(const spmvb200_cg_args_t &a, spmvb200_cg_result_t *out) {
    cudaStream_t s = static_cast<cudaStream_t>(a.stream);
    const int64_t n = a.n;
    const OffT *Ap = static_cast<const OffT *>(a.Ap);
    const ValT *Ax = static_cast<const ValT *>(a.Ax);
    const ValT *b = static_cast<const ValT *>(a.b);
    ValT *x = static_cast<ValT *>(a.x);

    unsigned grid = 0;
    SPMV_TRY(krylov_grid(n, &grid));

    // workspace: state | partials (3 sums per block) | r p q [z dinv]
    const size_t off_part = align256(sizeof(CgState));
    const size_t off_vec = off_part + align256((size_t)3 * grid * sizeof(double));
    const size_t vec = align256((size_t)n * sizeof(ValT));
    void *ws = nullptr;
    SPMV_TRY(scratch_get(s, SCRATCH_CG, off_vec + (kJacobi ? 5 : 3) * vec, &ws));
    char *base = static_cast<char *>(ws);
    CgState *st = reinterpret_cast<CgState *>(base);
    double *partial = reinterpret_cast<double *>(base + off_part);
    ValT *r = reinterpret_cast<ValT *>(base + off_vec);
    ValT *p = reinterpret_cast<ValT *>(base + off_vec + vec);
    ValT *q = reinterpret_cast<ValT *>(base + off_vec + 2 * vec);
    ValT *z = kJacobi ? reinterpret_cast<ValT *>(base + off_vec + 3 * vec) : r;
    ValT *dinv = kJacobi ? reinterpret_cast<ValT *>(base + off_vec + 4 * vec) : nullptr;

    SPMV_CUDA_TRY(cudaMemsetAsync(st, 0, sizeof(CgState), s));
    if (kJacobi) {
        jacobi_diag_kernel<OffT, ValT><<<grid, kKrylovBlock, 0, s>>>(n, Ap, a.Aj, Ax, dinv, &st->bad_diag);
        SPMV_LAUNCH_CHECK();
    }
    // r0 = b - A x0: the first SpMV on this matrix, so without the static-pattern flag
    SPMV_TRY(krylov_spmv(a, x, q, 0));
    cg_init_kernel<ValT, kJacobi><<<grid, kKrylovBlock, 0, s>>>(n, b, q, dinv, r, z, p, a.rtol, st, partial);
    SPMV_LAUNCH_CHECK();
    CgState h;
    SPMV_TRY(read_state(st, &h, s));
    if (h.bad_diag) return SPMVB200_ERR_INVALID;

    int64_t enqueued = 0, batch = 1;
    while (!h.converged && !h.breakdown && enqueued < a.max_iter) {
        const int64_t k = std::min(batch, a.max_iter - enqueued);
        for (int64_t it = 0; it < k; ++it) {
            SPMV_TRY(krylov_spmv(a, p, q, SPMVB200_FLAG_STATIC_PATTERN));
            cg_pq_kernel<ValT><<<grid, kKrylovBlock, 0, s>>>(n, p, q, st, partial);
            SPMV_LAUNCH_CHECK();
            cg_update_kernel<ValT, kJacobi><<<grid, kKrylovBlock, 0, s>>>(n, p, q, dinv, x, r, z, st, partial);
            SPMV_LAUNCH_CHECK();
            cg_direction_kernel<ValT><<<grid, kKrylovBlock, 0, s>>>(n, z, p, st);
            SPMV_LAUNCH_CHECK();
        }
        enqueued += k;
        batch = std::min(2 * batch, kKrylovMaxBatch);
        SPMV_TRY(read_state(st, &h, s));
    }
    // b = 0: the solution is x = 0, whatever x0 was
    if (h.bb == 0.0) SPMV_CUDA_TRY(cudaMemsetAsync(x, 0, (size_t)n * sizeof(ValT), s));
    krylov_residual_kernel<OffT, ValT><<<grid, kKrylovBlock, 0, s>>>(n, Ap, a.Aj, Ax, x, b, &st->res2, partial,
                                                                    &st->counter);
    SPMV_LAUNCH_CHECK();
    SPMV_TRY(read_state(st, &h, s));

    out->iterations = (int64_t)h.iterations;
    out->residual_norm = std::sqrt(h.res2);
    out->b_norm = std::sqrt(h.bb);
    out->converged = h.converged;
    out->breakdown = h.breakdown;
    return SPMVB200_OK;
}

}  // namespace

template <typename OffT, typename ValT>
int cg_solve(const spmvb200_cg_args_t &a, spmvb200_cg_result_t *out) {
    return (a.flags & SPMVB200_CG_JACOBI) ? cg_run<OffT, ValT, true>(a, out) : cg_run<OffT, ValT, false>(a, out);
}
template int cg_solve<int32_t, float>(const spmvb200_cg_args_t &, spmvb200_cg_result_t *);
template int cg_solve<int32_t, double>(const spmvb200_cg_args_t &, spmvb200_cg_result_t *);
template int cg_solve<int64_t, float>(const spmvb200_cg_args_t &, spmvb200_cg_result_t *);
template int cg_solve<int64_t, double>(const spmvb200_cg_args_t &, spmvb200_cg_result_t *);

}  // namespace spmvb200
