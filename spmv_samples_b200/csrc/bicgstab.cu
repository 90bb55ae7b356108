// bicgstab.cu -- right-preconditioned BiCGSTAB (van der Vorst) on a general square CSR matrix,
// with M = I or the Jacobi preconditioner M = diag(A), entirely on the device (spmvb200_bicgstab).
// The operations come in the order of scipy.sparse.linalg.bicgstab.
//
// One iteration is two SpMVs of the caller's kind (through spmvb200_spmv with
// SPMVB200_FLAG_STATIC_PATTERN) and five streaming kernels:
//   bicgstab_p_kernel      p = r + beta (p - omega v)  (p = r in the first iteration), p^ = dinv p
//   SpMV                   v = A p^
//   bicgstab_rv_kernel     (r^, v)                    -> alpha = rho / (r^, v)
//   bicgstab_s_kernel      s = r - alpha v, x += alpha p^, s^ = dinv s; ||s||^2
//                                                     -> iteration += 1, converged (half step)
//   SpMV                   t = A s^
//   bicgstab_omega_kernel  (t, s), (t, t)             -> omega = (t, s) / (t, t)
//   bicgstab_r_kernel      x += omega s^, r = s - omega t; (r^, r), ||r||^2
//                                                     -> converged, or rho, beta for the next one
// Without Jacobi p^ is p and s^ is s; s always lives in r's storage.  A breakdown is an exact zero
// or a non-finite value of rho, (r^, v), alpha, (t, t) or omega, or omega == 0 after the update;
// it leaves x at the last finite iterate.  Dot products accumulate in double in a fixed order
// (grid_sum, krylov.cuh); the scalars live in a device state block that the host reads once per
// batch of 1, 2, 4, ... kKrylovMaxBatch iterations.  Every kernel returns at once when
// `converged` or `breakdown` is set, so x and the iteration count do not depend on the batch
// boundaries (the SpMVs left in a batch still run; they only rewrite v and t).
#include <algorithm>
#include <cmath>

#include "krylov.cuh"

namespace spmvb200 {
namespace {

struct BicgState {
    double rho;    // (r^, r) of the current residual
    double alpha;  // rho / (r^, v)
    double omega;  // (t, s) / (t, t)
    double beta;   // (rho_new / rho) (alpha / omega)
    double bb;     // ||b||^2
    double tol;    // rtol * ||b||
    double res2;   // ||b - A x||^2 of the returned x, in fp64
    unsigned long long iterations;  // times x was moved by alpha p^
    int converged;
    int breakdown;
    int bad_diag;          // Jacobi: a row without a (non-zero) diagonal entry
    unsigned int counter;  // blocks finished in the running reduction; the last one resets it
};

__device__ __forceinline__ bool stopped(const BicgState *st) { return (st->converged | st->breakdown) != 0; }

// r = b - q (q = A x0), r^ = r; ||r||^2 (= rho), ||b||^2
template <typename ValT>
__global__ void __launch_bounds__(kKrylovBlock)
bicgstab_init_kernel(int64_t n, const ValT *__restrict__ b, const ValT *__restrict__ q, ValT *__restrict__ r,
                     ValT *__restrict__ rh, double rtol, BicgState *st, double *__restrict__ partial) {
    double acc[2] = {0.0, 0.0};  // r.r, b.b
    for (int64_t i = first_index(); i < n; i += grid_stride()) {
        const ValT bi = b[i];
        const ValT ri = bi - q[i];
        r[i] = ri;
        rh[i] = ri;
        acc[0] += (double)ri * (double)ri;
        acc[1] += (double)bi * (double)bi;
    }
    if (!grid_sum<2>(acc, partial, &st->counter)) return;
    if (threadIdx.x == 0) {
        const double rr = acc[0], bb = acc[1];
        st->rho = rr;
        st->bb = bb;
        st->tol = rtol * sqrt(bb);
        st->iterations = 0;
        if (bb == 0.0 || sqrt(rr) <= st->tol) st->converged = 1;
        else if (rr == 0.0 || !isfinite(rr)) st->breakdown = 1;
    }
}

// K1: p = r + beta (p - omega v), or p = r in the first iteration; p^ = dinv p
template <typename ValT, bool kJacobi>
__global__ void __launch_bounds__(kKrylovBlock)
bicgstab_p_kernel(int64_t n, const ValT *__restrict__ r, const ValT *__restrict__ v, const ValT *__restrict__ dinv,
                  ValT *__restrict__ p, ValT *__restrict__ ph, const BicgState *st) {
    if (stopped(st)) return;
    const bool first = st->iterations == 0;
    const ValT bt = (ValT)st->beta, om = (ValT)st->omega;
    for (int64_t i = first_index(); i < n; i += grid_stride()) {
        const ValT pi = first ? r[i] : r[i] + bt * (p[i] - om * v[i]);
        p[i] = pi;
        if (kJacobi) ph[i] = dinv[i] * pi;
    }
}

// K2: (r^, v) -> alpha
template <typename ValT>
__global__ void __launch_bounds__(kKrylovBlock)
bicgstab_rv_kernel(int64_t n, const ValT *__restrict__ rh, const ValT *__restrict__ v, BicgState *st,
                   double *__restrict__ partial) {
    if (stopped(st)) return;
    double acc[1] = {0.0};
    for (int64_t i = first_index(); i < n; i += grid_stride()) acc[0] += (double)rh[i] * (double)v[i];
    if (!grid_sum<1>(acc, partial, &st->counter)) return;
    if (threadIdx.x == 0) {
        const double rv = acc[0], alpha = st->rho / rv;
        if (rv == 0.0 || !isfinite(rv) || !isfinite(alpha)) st->breakdown = 1;
        else st->alpha = alpha;
    }
}

// K3: s = r - alpha v (in r's storage), x += alpha p^, s^ = dinv s; ||s||^2 -> one more
// iteration, converged at the half step
template <typename ValT, bool kJacobi>
__global__ void __launch_bounds__(kKrylovBlock)
bicgstab_s_kernel(int64_t n, const ValT *__restrict__ v, const ValT *__restrict__ ph, const ValT *__restrict__ dinv,
                  ValT *__restrict__ x, ValT *__restrict__ rs, ValT *__restrict__ sh, BicgState *st,
                  double *__restrict__ partial) {
    if (stopped(st)) return;
    const ValT a = (ValT)st->alpha;
    double acc[1] = {0.0};
    for (int64_t i = first_index(); i < n; i += grid_stride()) {
        const ValT si = rs[i] - a * v[i];
        rs[i] = si;
        x[i] += a * ph[i];
        if (kJacobi) sh[i] = dinv[i] * si;
        acc[0] += (double)si * (double)si;
    }
    if (!grid_sum<1>(acc, partial, &st->counter)) return;
    if (threadIdx.x == 0) {
        st->iterations += 1;
        if (sqrt(acc[0]) <= st->tol) st->converged = 1;
    }
}

// K4: (t, s) and (t, t) -> omega
template <typename ValT>
__global__ void __launch_bounds__(kKrylovBlock)
bicgstab_omega_kernel(int64_t n, const ValT *__restrict__ t, const ValT *__restrict__ s, BicgState *st,
                      double *__restrict__ partial) {
    if (stopped(st)) return;
    double acc[2] = {0.0, 0.0};  // t.s, t.t
    for (int64_t i = first_index(); i < n; i += grid_stride()) {
        const double ti = (double)t[i];
        acc[0] += ti * (double)s[i];
        acc[1] += ti * ti;
    }
    if (!grid_sum<2>(acc, partial, &st->counter)) return;
    if (threadIdx.x == 0) {
        const double tt = acc[1], omega = acc[0] / tt;
        if (tt == 0.0 || !isfinite(omega)) st->breakdown = 1;
        else st->omega = omega;
    }
}

// K5: x += omega s^, r = s - omega t (in place); (r^, r), ||r||^2 -> converged, or rho and beta
template <typename ValT, bool kJacobi>
__global__ void __launch_bounds__(kKrylovBlock)
bicgstab_r_kernel(int64_t n, const ValT *__restrict__ t, const ValT *__restrict__ sh, const ValT *__restrict__ rh,
                  ValT *__restrict__ x, ValT *__restrict__ rs, BicgState *st, double *__restrict__ partial) {
    if (stopped(st)) return;
    const ValT om = (ValT)st->omega;
    double acc[2] = {0.0, 0.0};  // r^.r, r.r
    for (int64_t i = first_index(); i < n; i += grid_stride()) {
        const ValT si = rs[i];
        x[i] += om * (kJacobi ? sh[i] : si);
        const ValT ri = si - om * t[i];
        rs[i] = ri;
        acc[0] += (double)rh[i] * (double)ri;
        acc[1] += (double)ri * (double)ri;
    }
    if (!grid_sum<2>(acc, partial, &st->counter)) return;
    if (threadIdx.x == 0) {
        const double rho = acc[0], rr = acc[1];
        if (sqrt(rr) <= st->tol) {
            st->converged = 1;
        } else if (st->omega == 0.0 || rho == 0.0 || !isfinite(rho)) {
            st->breakdown = 1;
        } else {
            st->beta = (rho / st->rho) * (st->alpha / st->omega);
            st->rho = rho;
        }
    }
}

template <typename OffT, typename ValT, bool kJacobi>
int bicgstab_run(const spmvb200_cg_args_t &a, spmvb200_cg_result_t *out) {
    cudaStream_t s = static_cast<cudaStream_t>(a.stream);
    const int64_t n = a.n;
    const OffT *Ap = static_cast<const OffT *>(a.Ap);
    const ValT *Ax = static_cast<const ValT *>(a.Ax);
    const ValT *b = static_cast<const ValT *>(a.b);
    ValT *x = static_cast<ValT *>(a.x);

    unsigned grid = 0;
    SPMV_TRY(krylov_grid(n, &grid));

    // workspace: state | partials (2 sums per block) | r(s) r^ p v t [p^ s^ dinv]
    const size_t off_part = align256(sizeof(BicgState));
    const size_t off_vec = off_part + align256((size_t)2 * grid * sizeof(double));
    const size_t vec = align256((size_t)n * sizeof(ValT));
    void *ws = nullptr;
    SPMV_TRY(scratch_get(s, SCRATCH_BICGSTAB, off_vec + (kJacobi ? 8 : 5) * vec, &ws));
    char *base = static_cast<char *>(ws);
    BicgState *st = reinterpret_cast<BicgState *>(base);
    double *partial = reinterpret_cast<double *>(base + off_part);
    ValT *vecs[8];
    for (int k = 0; k < (kJacobi ? 8 : 5); ++k) vecs[k] = reinterpret_cast<ValT *>(base + off_vec + k * vec);
    ValT *r = vecs[0], *rh = vecs[1], *p = vecs[2], *v = vecs[3], *t = vecs[4];
    ValT *ph = kJacobi ? vecs[5] : p;
    ValT *sh = kJacobi ? vecs[6] : r;
    ValT *dinv = kJacobi ? vecs[7] : nullptr;

    SPMV_CUDA_TRY(cudaMemsetAsync(st, 0, sizeof(BicgState), s));
    if (kJacobi) {
        jacobi_diag_kernel<OffT, ValT><<<grid, kKrylovBlock, 0, s>>>(n, Ap, a.Aj, Ax, dinv, &st->bad_diag);
        SPMV_LAUNCH_CHECK();
    }
    // r0 = b - A x0: the first SpMV on this matrix, so without the static-pattern flag
    SPMV_TRY(krylov_spmv(a, x, v, 0));
    bicgstab_init_kernel<ValT><<<grid, kKrylovBlock, 0, s>>>(n, b, v, r, rh, a.rtol, st, partial);
    SPMV_LAUNCH_CHECK();
    BicgState h;
    SPMV_TRY(read_state(st, &h, s));
    if (h.bad_diag) return SPMVB200_ERR_INVALID;

    int64_t enqueued = 0, batch = 1;
    while (!h.converged && !h.breakdown && enqueued < a.max_iter) {
        const int64_t k = std::min(batch, a.max_iter - enqueued);
        for (int64_t it = 0; it < k; ++it) {
            bicgstab_p_kernel<ValT, kJacobi><<<grid, kKrylovBlock, 0, s>>>(n, r, v, dinv, p, ph, st);
            SPMV_LAUNCH_CHECK();
            SPMV_TRY(krylov_spmv(a, ph, v, SPMVB200_FLAG_STATIC_PATTERN));
            bicgstab_rv_kernel<ValT><<<grid, kKrylovBlock, 0, s>>>(n, rh, v, st, partial);
            SPMV_LAUNCH_CHECK();
            bicgstab_s_kernel<ValT, kJacobi><<<grid, kKrylovBlock, 0, s>>>(n, v, ph, dinv, x, r, sh, st, partial);
            SPMV_LAUNCH_CHECK();
            SPMV_TRY(krylov_spmv(a, sh, t, SPMVB200_FLAG_STATIC_PATTERN));
            bicgstab_omega_kernel<ValT><<<grid, kKrylovBlock, 0, s>>>(n, t, r, st, partial);
            SPMV_LAUNCH_CHECK();
            bicgstab_r_kernel<ValT, kJacobi><<<grid, kKrylovBlock, 0, s>>>(n, t, sh, rh, x, r, st, partial);
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
int bicgstab_solve(const spmvb200_cg_args_t &a, spmvb200_cg_result_t *out) {
    return (a.flags & SPMVB200_CG_JACOBI) ? bicgstab_run<OffT, ValT, true>(a, out)
                                          : bicgstab_run<OffT, ValT, false>(a, out);
}
template int bicgstab_solve<int32_t, float>(const spmvb200_cg_args_t &, spmvb200_cg_result_t *);
template int bicgstab_solve<int32_t, double>(const spmvb200_cg_args_t &, spmvb200_cg_result_t *);
template int bicgstab_solve<int64_t, float>(const spmvb200_cg_args_t &, spmvb200_cg_result_t *);
template int bicgstab_solve<int64_t, double>(const spmvb200_cg_args_t &, spmvb200_cg_result_t *);

}  // namespace spmvb200
