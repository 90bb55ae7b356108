// krylov.cuh -- pieces the device-resident Krylov solvers (cg.cu, bicgstab.cu, gmres.cu) share:
// the fixed-order fp64 block and grid reductions, the Jacobi diagonal, the fp64 true residual,
// the SpMV call on the solver's arguments and the read of a solver's device state block.
//
// Every dot product accumulates in double in a fixed order: per-block partials, then the last
// block to finish (threadfence + counter, as norm_exchange_kernel in power.cu) adds them in block
// order.  So a solve is deterministic for the deterministic SpMV kinds.
#pragma once

#include <algorithm>
#include <cstring>

#include "common.cuh"

namespace spmvb200 {

constexpr int kKrylovBlock = 256;
constexpr int kKrylovBlocksPerSm = 8;
constexpr int64_t kKrylovMaxBatch = 64;  // iterations enqueued between two reads of the flags, at most

// N block sums in a fixed order; the totals are valid in thread 0
template <int N>
__device__ __forceinline__ void block_sum(double (&v)[N]) {
    __shared__ double s[N][kKrylovBlock / 32];
#pragma unroll
    for (int j = 0; j < N; ++j) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v[j] += __shfl_xor_sync(0xffffffffu, v[j], d);
        if ((threadIdx.x & 31) == 0) s[j][threadIdx.x >> 5] = v[j];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int j = 0; j < N; ++j) {
            double t = 0.0;
#pragma unroll
            for (int w = 0; w < kKrylovBlock / 32; ++w) t += s[j][w];
            v[j] = t;
        }
    }
    __syncthreads();  // s may be reused
}

// Grid-wide sums of v: true in the last block to finish, whose thread 0 then holds the totals,
// added in block order (the same bits on every run with the same grid).
template <int N>
__device__ __forceinline__ bool grid_sum(double (&v)[N], double *partial, unsigned int *counter) {
    __shared__ bool is_last;
    block_sum<N>(v);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int j = 0; j < N; ++j) partial[(size_t)j * gridDim.x + blockIdx.x] = v[j];
        __threadfence();
        is_last = atomicAdd(counter, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!is_last) return false;
    __threadfence();
#pragma unroll
    for (int j = 0; j < N; ++j) {
        v[j] = 0.0;
        for (int i = threadIdx.x; i < (int)gridDim.x; i += kKrylovBlock) v[j] += __ldcg(partial + (size_t)j * gridDim.x + i);
    }
    block_sum<N>(v);
    if (threadIdx.x == 0) *counter = 0;  // ready for the next reduction
    return true;
}

// Sums whose count is known only at run time (GMRES: one dot product per basis vector).  Each
// warp adds its lanes' terms in the shuffle order of block_sum and keeps a running total per sum
// in shared memory, s[c * kKrylovWarps + warp]; grid_sum_n then adds the warps in order, writes
// one partial per block and sum, and the last block to finish adds the partials in block order,
// as grid_sum does.  Every thread of the block calls both, with warp-uniform control flow.
constexpr int kKrylovWarps = kKrylovBlock / 32;

__device__ __forceinline__ void warp_accumulate(double v, double *s_c) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    if ((threadIdx.x & 31) == 0) s_c[threadIdx.x >> 5] += v;
}

// The `count` totals of the running warp sums in s: true in the last block to finish, where
// tot[0 .. count) (shared) then holds them for every thread.  s is overwritten.
__device__ __forceinline__ bool grid_sum_n(int count, double *s, double *tot, double *partial,
                                           unsigned int *counter) {
    __shared__ bool is_last;
    __syncthreads();
    for (int c = threadIdx.x; c < count; c += kKrylovBlock) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kKrylovWarps; ++w) t += s[c * kKrylovWarps + w];
        partial[(size_t)c * gridDim.x + blockIdx.x] = t;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = atomicAdd(counter, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!is_last) return false;
    __threadfence();
    for (int c = 0; c < count; ++c) {
        double v = 0.0;
        for (int i = threadIdx.x; i < (int)gridDim.x; i += kKrylovBlock) v += __ldcg(partial + (size_t)c * gridDim.x + i);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
        if ((threadIdx.x & 31) == 0) s[c * kKrylovWarps + (threadIdx.x >> 5)] = v;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < count; c += kKrylovBlock) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kKrylovWarps; ++w) t += s[c * kKrylovWarps + w];
        tot[c] = t;
    }
    __syncthreads();
    if (threadIdx.x == 0) *counter = 0;  // ready for the next reduction
    return true;
}

__device__ __forceinline__ int64_t first_index() { return (int64_t)blockIdx.x * kKrylovBlock + threadIdx.x; }
__device__ __forceinline__ int64_t grid_stride() { return (int64_t)gridDim.x * kKrylovBlock; }

// dinv[i] = 1 / A[i,i]: row i searched for column i (duplicates are added, as the SpMV adds them);
// *bad_diag = 1 for a row without a (non-zero) diagonal entry
template <typename OffT, typename ValT>
__global__ void __launch_bounds__(kKrylovBlock)
jacobi_diag_kernel(int64_t n, const OffT *__restrict__ Ap, const int32_t *__restrict__ Aj,
                   const ValT *__restrict__ Ax, ValT *__restrict__ dinv, int *bad_diag) {
    for (int64_t i = first_index(); i < n; i += grid_stride()) {
        double d = 0.0;
        bool found = false;
        for (OffT k = Ap[i]; k < Ap[i + 1]; ++k) {
            if (Aj[k] == (int32_t)i) {
                d += (double)Ax[k];
                found = true;
            }
        }
        const bool ok = found && d != 0.0;
        if (!ok) *bad_diag = 1;
        dinv[i] = ok ? (ValT)(1.0 / d) : ValT(0);
    }
}

// *res2 = ||b - A x||^2 in fp64, one row per thread: products and sums in double, in row order,
// without contraction -- per row the same operations as the fp64 host reference, for both value
// types
template <typename OffT, typename ValT>
__global__ void __launch_bounds__(kKrylovBlock)
krylov_residual_kernel(int64_t n, const OffT *__restrict__ Ap, const int32_t *__restrict__ Aj,
                       const ValT *__restrict__ Ax, const ValT *__restrict__ x, const ValT *__restrict__ b,
                       double *res2, double *__restrict__ partial, unsigned int *counter) {
    double acc[1] = {0.0};
    for (int64_t i = first_index(); i < n; i += grid_stride()) {
        double y = 0.0;
        for (OffT k = Ap[i]; k < Ap[i + 1]; ++k) y = __dadd_rn(y, __dmul_rn((double)Ax[k], (double)x[Aj[k]]));
        const double ri = __dsub_rn((double)b[i], y);
        acc[0] += ri * ri;
    }
    if (!grid_sum<1>(acc, partial, counter)) return;
    if (threadIdx.x == 0) *res2 = acc[0];
}

inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

// blocks of a solver's streaming kernels: one element per thread, at most kKrylovBlocksPerSm per SM
inline int krylov_grid(int64_t n, unsigned *grid) {
    const DeviceInfo *di = nullptr;
    SPMV_TRY(current_device_info(&di));
    const int64_t cap = (int64_t)di->sm_count * kKrylovBlocksPerSm;
    *grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + kKrylovBlock - 1) / kKrylovBlock, cap));
    return SPMVB200_OK;
}

// out = A in, with the solver's kind and matrix
inline int krylov_spmv(const spmvb200_cg_args_t &a, const void *in, void *out, int flags) {
    spmvb200_args_t s;
    std::memset(&s, 0, sizeof(s));
    s.kind = a.kind;
    s.offset_bits = a.offset_bits;
    s.value_bits = a.value_bits;
    s.n_rows = s.n_cols = a.n;
    s.nnz = a.nnz;
    s.Ap = a.Ap;
    s.Aj = a.Aj;
    s.Ax = a.Ax;
    s.x = in;
    s.y = out;
    s.stream = a.stream;
    s.flags = flags;
    return spmvb200_spmv(&s);
}

// the solver's device state block, copied to the host once the stream has reached this point
template <typename State>
int read_state(const State *st_dev, State *h, cudaStream_t stream) {
    SPMV_CUDA_TRY(cudaMemcpyAsync(h, st_dev, sizeof(State), cudaMemcpyDeviceToHost, stream));
    SPMV_CUDA_TRY(cudaStreamSynchronize(stream));
    return SPMVB200_OK;
}

}  // namespace spmvb200
