// gmres.cu -- right-preconditioned restarted GMRES(m) on a general square CSR matrix, with M = I
// or the Jacobi preconditioner M = diag(A), entirely on the device (spmvb200_gmres).
//
// A cycle builds an orthonormal basis V = [v_0 .. v_k] of the Krylov space of A M^-1 from
// v_0 = r / ||r||, r = b - A x the true residual, and ends with x += M^-1 V y, y minimising
// ||beta e_1 - H y|| (H the Hessenberg matrix of the Arnoldi relation).  With right
// preconditioning that is the true residual, so rtol means what it means for cg and bicgstab.
// One Arnoldi step j is one SpMV of the caller's kind (SPMVB200_FLAG_STATIC_PATTERN) and four
// streaming kernels, whatever j is:
//   SpMV                    w = A z_j, into v_{j+1}'s storage  (z_j = v_j, or dinv v_j)
//   gmres_dot_kernel        h1 = V^T w, ||w||^2                       (classical Gram-Schmidt ...
//   gmres_orth_dot_kernel   w -= V h1; h2 = V^T w                      ... with one re-
//   gmres_orth_norm_kernel  w -= V h2; ||w||^2 -> H[:, j] = h1 + h2,   orthogonalisation: CGS2)
//                           the Givens rotations, the residual estimate |g_{j+1}|, the cycle end
//   gmres_scale_kernel      v_{j+1} = w / ||w||, z_{j+1} = dinv v_{j+1}
// and a cycle ends with
//   gmres_x_kernel          x += M^-1 (V y)                   (y solved by the step that ended it)
//   SpMV                    q = A x, into v_0's storage
//   gmres_residual_kernel   r = b - q, ||r||^2 (and ||b||^2) -> converged, breakdown or next cycle
//   gmres_scale_kernel      v_0 = r / ||r||
// The set-up is the same as a cycle end without the x update.  The rotations use
// r = hypot(a, b), c = a / r, s = b / r (c = 1, s = 0 at r = 0), so g_{j+1} = -s g_j.  A cycle
// ends after m steps, when |g_{j+1}| <= rtol ||b||, at a lucky breakdown (||w|| after the
// orthogonalisation <= eps ||w|| before it, eps of the value type: v_{j+1} is not formed), or at
// the step cap; the explicit ||r|| then decides convergence.  A lucky breakdown whose explicit
// residual misses the tolerance, a non-finite h, norm or rotation (x stays at the start of the
// cycle), or a non-finite ||b|| or ||r0|| is a breakdown.
//
// Batching: the host enqueues step slots in batches of 1, 2, 4, ... kKrylovMaxBatch and reads the
// state block after each batch.  Cycles are aligned to slots: the host enqueues a cycle end after
// every m-th slot and after slot max_iter, and a cycle that ended early on the device leaves its
// remaining slots idle (every kernel returns at once; the SpMVs still run and only write basis
// columns past the ones the cycle used).  So x, `iterations` and the flags do not depend on the
// batch boundaries.  Launches, for S enqueued slots and C = ceil(S / m) cycle ends: the set-up
// (Jacobi diagonal, one SpMV, two kernels), S times (one SpMV + 4 kernels), C times (one SpMV + 3
// kernels) and the final fp64 residual kernel.  S is at most max_iter, and past the slot where
// the solve stopped, at most one batch (kKrylovMaxBatch slots) more.
#include <algorithm>
#include <cfloat>
#include <cmath>

#include "krylov.cuh"

namespace spmvb200 {
namespace {

constexpr int kMaxM = SPMVB200_GMRES_MAX_RESTART;
constexpr int kMaxSums = kMaxM + 2;  // h1: one dot per basis vector and ||w||^2

struct GmresState {
    double H[kMaxM][kMaxM + 1];  // column j of the rotated Hessenberg matrix, rows 0 .. j
    double cs[kMaxM], sn[kMaxM];  // the Givens rotations of the cycle
    double g[kMaxM + 1];         // rotated beta e_1; |g[k]| estimates ||r|| after k steps
    double y[kMaxM];             // the cycle's minimiser, solved by the step that ended it
    double h1[kMaxM + 2];        // V^T w of the first pass; [k + 1] = ||w||^2 before it
    double h2[kMaxM + 1];        // V^T w of the second pass
    double bb;                   // ||b||^2
    double tol;                  // rtol * ||b||
    double scale;                // 1 / norm of the basis column gmres_scale_kernel normalises
    double res2;                 // ||b - A x||^2 of the returned x, in fp64
    unsigned long long iterations;  // Arnoldi steps completed, over all cycles
    int k;                       // steps completed in this cycle: basis columns 0 .. k exist
    int active;                  // the cycle takes more steps
    int lucky;                   // the cycle ended at a lucky breakdown
    int started;                 // the set-up's residual has been taken
    int converged;
    int breakdown;
    int bad_diag;                // Jacobi: a row without a (non-zero) diagonal entry
    unsigned int counter;        // blocks finished in the running reduction; the last one resets it
};

__device__ __forceinline__ bool stopped(const GmresState *st) { return (st->converged | st->breakdown) != 0; }

template <typename ValT>
__device__ __forceinline__ double value_eps() { return sizeof(ValT) == 4 ? (double)FLT_EPSILON : DBL_EPSILON; }

// zero the running warp sums of `count` sums
__device__ __forceinline__ void zero_sums(double *s, int count) {
    for (int i = threadIdx.x; i < count * kKrylovWarps; i += kKrylovBlock) s[i] = 0.0;
    __syncthreads();
}

// the loops below walk the grid-stride range a warp at a time, so that every lane of a warp
// takes part in its shuffles; `i < n` masks the tail
__device__ __forceinline__ int64_t warp_first_index() { return first_index() - (threadIdx.x & 31); }

// y from R y = g (k x k upper triangular), back substitution in the order of
// scipy.sparse.linalg.gmres, which also pseudo-solves a zero last diagonal entry
__device__ void solve_y(GmresState *st, int k) {
    double *y = st->y;
    for (int i = 0; i < k; ++i) y[i] = st->g[i];
    if (st->H[k - 1][k - 1] == 0.0) y[k - 1] = 0.0;
    for (int i = k - 1; i > 0; --i) {
        if (y[i] != 0.0) {
            y[i] /= st->H[i][i];
            const double t = y[i];
            for (int l = 0; l < i; ++l) y[l] -= t * st->H[i][l];
        }
    }
    if (y[0] != 0.0) y[0] /= st->H[0][0];
}

// K1: h1 = V^T w (w = column k + 1, V = columns 0 .. k), ||w||^2
template <typename ValT>
__global__ void __launch_bounds__(kKrylovBlock)
gmres_dot_kernel(int64_t n, const ValT *__restrict__ V, int64_t ldv, GmresState *st, double *__restrict__ partial) {
    __shared__ double s[kMaxSums * kKrylovWarps];
    __shared__ double tot[kMaxSums];
    if (!st->active) return;
    const int k = st->k;
    const ValT *w = V + (k + 1) * ldv;
    zero_sums(s, k + 2);
    for (int64_t base = warp_first_index(); base < n; base += grid_stride()) {
        const int64_t i = base + (threadIdx.x & 31);
        const bool in = i < n;
        const double wi = in ? (double)w[i] : 0.0;
#pragma unroll 4
        for (int c = 0; c <= k; ++c) warp_accumulate(in ? (double)V[c * ldv + i] * wi : 0.0, s + c * kKrylovWarps);
        warp_accumulate(wi * wi, s + (k + 1) * kKrylovWarps);
    }
    if (!grid_sum_n(k + 2, s, tot, partial, &st->counter)) return;
    for (int c = threadIdx.x; c < k + 2; c += kKrylovBlock) st->h1[c] = tot[c];
}

// K2: w -= V h1, then h2 = V^T w on the updated w, in the same pass
template <typename ValT>
__global__ void __launch_bounds__(kKrylovBlock)
gmres_orth_dot_kernel(int64_t n, ValT *__restrict__ V, int64_t ldv, GmresState *st, double *__restrict__ partial) {
    __shared__ double s[kMaxSums * kKrylovWarps];
    __shared__ double tot[kMaxSums];
    __shared__ ValT h[kMaxM];
    if (!st->active) return;
    const int k = st->k;
    ValT *w = V + (k + 1) * ldv;
    for (int c = threadIdx.x; c <= k; c += kKrylovBlock) h[c] = (ValT)st->h1[c];
    zero_sums(s, k + 1);
    for (int64_t base = warp_first_index(); base < n; base += grid_stride()) {
        const int64_t i = base + (threadIdx.x & 31);
        const bool in = i < n;
        ValT wi = ValT(0);
        if (in) {
            wi = w[i];
            for (int c = 0; c <= k; ++c) wi -= h[c] * V[c * ldv + i];
            w[i] = wi;
        }
        const double wd = (double)wi;
#pragma unroll 4
        for (int c = 0; c <= k; ++c) warp_accumulate(in ? (double)V[c * ldv + i] * wd : 0.0, s + c * kKrylovWarps);
    }
    if (!grid_sum_n(k + 1, s, tot, partial, &st->counter)) return;
    for (int c = threadIdx.x; c <= k; c += kKrylovBlock) st->h2[c] = tot[c];
}

// after step k: H[:, k] = h1 + h2 and ||w||; the earlier rotations, a new one, the residual
// estimate; the cycle's end (solving y) or the scale of v_{k+1}.  One thread.
template <typename ValT>
__device__ void arnoldi_update(GmresState *st, int k, double ww, bool last_slot) {
    double *col = st->H[k];
    bool finite = true;
    for (int i = 0; i <= k; ++i) {
        col[i] = st->h1[i] + st->h2[i];
        finite &= isfinite(col[i]);
    }
    const double h0 = sqrt(st->h1[k + 1]);
    double hn = sqrt(ww);
    finite &= isfinite(h0) && isfinite(hn);
    const bool lucky = hn <= value_eps<ValT>() * h0;
    if (lucky) hn = 0.0;
    for (int i = 0; i < k; ++i) {
        const double c = st->cs[i], s = st->sn[i], n0 = col[i], n1 = col[i + 1];
        col[i] = c * n0 + s * n1;
        col[i + 1] = -s * n0 + c * n1;
    }
    const double a = col[k], r = hypot(a, hn);
    const double c = r == 0.0 ? 1.0 : a / r, s = r == 0.0 ? 0.0 : hn / r;
    col[k] = r;
    st->cs[k] = c;
    st->sn[k] = s;
    const double gk = st->g[k], gk1 = -s * gk;
    for (int i = 0; i < k; ++i) finite &= isfinite(col[i]);
    finite &= isfinite(r) && isfinite(c) && isfinite(s) && isfinite(gk1);
    if (!finite) {  // x stays at the start of the cycle
        st->breakdown = 1;
        st->active = 0;
        return;
    }
    st->g[k] = c * gk;
    st->g[k + 1] = gk1;
    st->iterations += 1;
    st->k = k + 1;
    if (lucky || fabs(gk1) <= st->tol || last_slot) {
        st->active = 0;
        st->lucky = lucky;
        solve_y(st, k + 1);
    } else {
        st->scale = 1.0 / hn;
    }
}

// K3: w -= V h2; ||w||^2 -> arnoldi_update
template <typename ValT>
__global__ void __launch_bounds__(kKrylovBlock)
gmres_orth_norm_kernel(int64_t n, ValT *__restrict__ V, int64_t ldv, int last_slot, GmresState *st,
                       double *__restrict__ partial) {
    __shared__ double s[kKrylovWarps];
    __shared__ double tot[1];
    __shared__ ValT h[kMaxM];
    if (!st->active) return;
    const int k = st->k;
    ValT *w = V + (k + 1) * ldv;
    for (int c = threadIdx.x; c <= k; c += kKrylovBlock) h[c] = (ValT)st->h2[c];
    zero_sums(s, 1);
    for (int64_t base = warp_first_index(); base < n; base += grid_stride()) {
        const int64_t i = base + (threadIdx.x & 31);
        const bool in = i < n;
        ValT wi = ValT(0);
        if (in) {
            wi = w[i];
#pragma unroll 4
            for (int c = 0; c <= k; ++c) wi -= h[c] * V[c * ldv + i];
            w[i] = wi;
        }
        warp_accumulate((double)wi * (double)wi, s);
    }
    if (!grid_sum_n(1, s, tot, partial, &st->counter)) return;
    if (threadIdx.x == 0) arnoldi_update<ValT>(st, k, tot[0], last_slot != 0);
}

// K4: v_k *= scale (k = 0 at a cycle's start), z = dinv v_k
template <typename ValT, bool kJacobi>
__global__ void __launch_bounds__(kKrylovBlock)
gmres_scale_kernel(int64_t n, ValT *__restrict__ V, int64_t ldv, const ValT *__restrict__ dinv, ValT *__restrict__ z,
                   const GmresState *st) {
    if (!st->active) return;
    ValT *v = V + st->k * ldv;
    const ValT sc = (ValT)st->scale;
    for (int64_t i = first_index(); i < n; i += grid_stride()) {
        const ValT vi = v[i] * sc;
        v[i] = vi;
        if (kJacobi) z[i] = dinv[i] * vi;
    }
}

// cycle end: x += M^-1 (V y), V y summed in double in column order
template <typename ValT, bool kJacobi>
__global__ void __launch_bounds__(kKrylovBlock)
gmres_x_kernel(int64_t n, const ValT *__restrict__ V, int64_t ldv, const ValT *__restrict__ dinv, ValT *__restrict__ x,
               const GmresState *st) {
    __shared__ double y[kMaxM];
    if (stopped(st) || st->k == 0) return;
    const int k = st->k;
    for (int c = threadIdx.x; c < k; c += kKrylovBlock) y[c] = st->y[c];
    __syncthreads();
    for (int64_t i = first_index(); i < n; i += grid_stride()) {
        double u = 0.0;
#pragma unroll 4
        for (int c = 0; c < k; ++c) u += y[c] * (double)V[c * ldv + i];
        x[i] += (ValT)(kJacobi ? (double)dinv[i] * u : u);
    }
}

// set-up and cycle end: r = b - q (q = A x, r in q's storage); ||r||^2, ||b||^2 -> converged,
// breakdown, or the next cycle from v_0 = r / ||r||
template <typename ValT>
__global__ void __launch_bounds__(kKrylovBlock)
gmres_residual_kernel(int64_t n, const ValT *__restrict__ b, ValT *__restrict__ qr, double rtol, GmresState *st,
                      double *__restrict__ partial) {
    if (stopped(st)) return;
    double acc[2] = {0.0, 0.0};  // r.r, b.b
    for (int64_t i = first_index(); i < n; i += grid_stride()) {
        const ValT bi = b[i];
        const ValT ri = bi - qr[i];
        qr[i] = ri;
        acc[0] += (double)ri * (double)ri;
        acc[1] += (double)bi * (double)bi;
    }
    if (!grid_sum<2>(acc, partial, &st->counter)) return;
    if (threadIdx.x == 0) {
        const double rr = acc[0], rn = sqrt(rr);
        if (!st->started) {
            st->started = 1;
            st->bb = acc[1];
            st->tol = rtol * sqrt(acc[1]);
            if (st->bb == 0.0 || rn <= st->tol) st->converged = 1;
            else if (!isfinite(st->bb) || !isfinite(rr)) st->breakdown = 1;
        } else if (rn <= st->tol) {
            st->converged = 1;
        } else if (st->lucky || !isfinite(rr)) {
            st->breakdown = 1;
        }
        if (!stopped(st)) {
            st->active = 1;
            st->k = 0;
            st->lucky = 0;
            st->g[0] = rn;
            st->scale = 1.0 / rn;
        }
    }
}

template <typename OffT, typename ValT, bool kJacobi>
int gmres_run(const spmvb200_cg_args_t &a, int restart, spmvb200_cg_result_t *out) {
    cudaStream_t s = static_cast<cudaStream_t>(a.stream);
    const int64_t n = a.n;
    const int m = (int)std::min<int64_t>(restart, n);
    const OffT *Ap = static_cast<const OffT *>(a.Ap);
    const ValT *Ax = static_cast<const ValT *>(a.Ax);
    const ValT *b = static_cast<const ValT *>(a.b);
    ValT *x = static_cast<ValT *>(a.x);

    unsigned grid = 0;
    SPMV_TRY(krylov_grid(n, &grid));

    // workspace: state | partials (m + 2 sums per block) | V: m + 1 columns [z dinv]
    const size_t off_part = align256(sizeof(GmresState));
    const size_t off_vec = off_part + align256((size_t)(m + 2) * grid * sizeof(double));
    const size_t vec = align256((size_t)n * sizeof(ValT));
    const int64_t ldv = (int64_t)(vec / sizeof(ValT));
    void *ws = nullptr;
    SPMV_TRY(scratch_get(s, SCRATCH_GMRES, off_vec + (m + 1 + (kJacobi ? 2 : 0)) * vec, &ws));
    char *base = static_cast<char *>(ws);
    GmresState *st = reinterpret_cast<GmresState *>(base);
    double *partial = reinterpret_cast<double *>(base + off_part);
    ValT *V = reinterpret_cast<ValT *>(base + off_vec);
    ValT *z = kJacobi ? V + (m + 1) * ldv : nullptr;
    ValT *dinv = kJacobi ? V + (m + 2) * ldv : nullptr;

    // r = b - A x into v_0, its norm deciding convergence or the next cycle, v_0 normalised
    auto restart_from_x = [&](int flags) -> int {
        SPMV_TRY(krylov_spmv(a, x, V, flags));
        gmres_residual_kernel<ValT><<<grid, kKrylovBlock, 0, s>>>(n, b, V, a.rtol, st, partial);
        SPMV_LAUNCH_CHECK();
        gmres_scale_kernel<ValT, kJacobi><<<grid, kKrylovBlock, 0, s>>>(n, V, ldv, dinv, z, st);
        SPMV_LAUNCH_CHECK();
        return SPMVB200_OK;
    };

    SPMV_CUDA_TRY(cudaMemsetAsync(st, 0, sizeof(GmresState), s));
    if (kJacobi) {
        jacobi_diag_kernel<OffT, ValT><<<grid, kKrylovBlock, 0, s>>>(n, Ap, a.Aj, Ax, dinv, &st->bad_diag);
        SPMV_LAUNCH_CHECK();
    }
    // the first SpMV on this matrix, so without the static-pattern flag
    SPMV_TRY(restart_from_x(0));
    GmresState h;
    SPMV_TRY(read_state(st, &h, s));
    if (h.bad_diag) return SPMVB200_ERR_INVALID;

    int64_t enqueued = 0, batch = 1;
    while (!h.converged && !h.breakdown && enqueued < a.max_iter) {
        const int64_t k = std::min(batch, a.max_iter - enqueued);
        for (int64_t it = 0; it < k; ++it) {
            const int64_t j = enqueued % m;  // the slot's step within its cycle
            const bool last = j == m - 1 || enqueued + 1 == a.max_iter;
            SPMV_TRY(krylov_spmv(a, kJacobi ? z : V + j * ldv, V + (j + 1) * ldv, SPMVB200_FLAG_STATIC_PATTERN));
            gmres_dot_kernel<ValT><<<grid, kKrylovBlock, 0, s>>>(n, V, ldv, st, partial);
            SPMV_LAUNCH_CHECK();
            gmres_orth_dot_kernel<ValT><<<grid, kKrylovBlock, 0, s>>>(n, V, ldv, st, partial);
            SPMV_LAUNCH_CHECK();
            gmres_orth_norm_kernel<ValT><<<grid, kKrylovBlock, 0, s>>>(n, V, ldv, last ? 1 : 0, st, partial);
            SPMV_LAUNCH_CHECK();
            gmres_scale_kernel<ValT, kJacobi><<<grid, kKrylovBlock, 0, s>>>(n, V, ldv, dinv, z, st);
            SPMV_LAUNCH_CHECK();
            ++enqueued;
            if (last) {
                gmres_x_kernel<ValT, kJacobi><<<grid, kKrylovBlock, 0, s>>>(n, V, ldv, dinv, x, st);
                SPMV_LAUNCH_CHECK();
                SPMV_TRY(restart_from_x(SPMVB200_FLAG_STATIC_PATTERN));
            }
        }
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
int gmres_solve(const spmvb200_cg_args_t &a, int restart, spmvb200_cg_result_t *out) {
    return (a.flags & SPMVB200_CG_JACOBI) ? gmres_run<OffT, ValT, true>(a, restart, out)
                                          : gmres_run<OffT, ValT, false>(a, restart, out);
}
template int gmres_solve<int32_t, float>(const spmvb200_cg_args_t &, int, spmvb200_cg_result_t *);
template int gmres_solve<int32_t, double>(const spmvb200_cg_args_t &, int, spmvb200_cg_result_t *);
template int gmres_solve<int64_t, float>(const spmvb200_cg_args_t &, int, spmvb200_cg_result_t *);
template int gmres_solve<int64_t, double>(const spmvb200_cg_args_t &, int, spmvb200_cg_result_t *);

}  // namespace spmvb200
