// common.cuh -- shared host/device plumbing of libspmvb200 (sm_100a only).
//
// Replaces reference/include/common.cuh:1-23 (checkCudaErr -> abort) with status codes,
// and holds the PTX wrappers the three kernels share: mbarrier + cp.async.bulk (TMA 1-D
// bulk copies, SASS UBLKCP), L2 cache-policy loads, and warp reductions.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>

#include "../../include/spmv_b200.h"

namespace spmvb200 {

// ------------------------------------------------------------------ host: status + errors
void record_cuda_error(cudaError_t e, const char *what, const char *file, int line);
void count_launch(int n = 1);

#define SPMV_CUDA_TRY(expr)                                                    \
    do {                                                                       \
        cudaError_t _e = (expr);                                               \
        if (_e != cudaSuccess) {                                               \
            ::spmvb200::record_cuda_error(_e, #expr, __FILE__, __LINE__);      \
            return SPMVB200_ERR_CUDA;                                          \
        }                                                                      \
    } while (0)

#define SPMV_TRY(expr)                          \
    do {                                        \
        int _s = (expr);                        \
        if (_s != SPMVB200_OK) return _s;       \
    } while (0)

// after a kernel launch
#define SPMV_LAUNCH_CHECK()                     \
    do {                                        \
        ::spmvb200::count_launch();             \
        SPMV_CUDA_TRY(cudaGetLastError());      \
    } while (0)

struct DeviceInfo {
    int device = -1;
    int sm_count = 0;
    int max_threads_per_sm = 0;
    size_t l2_bytes = 0;
    size_t persisting_l2_max = 0;
    size_t access_window_max = 0;
    size_t smem_optin = 0;
};
int current_device_info(const DeviceInfo **out);

// cudaFuncAttributePreferredSharedMemoryCarveout for `kernel` on the current device, applied
// once per (device, kernel, value).  percent < 0 = the driver's default.
int apply_max_dynamic_smem(const void *kernel, int64_t bytes);
int apply_carveout(const void *kernel, int64_t percent);

// Per-(device, stream) scratch that survives across calls, grown on demand.
// Slots keep independent buffers so a kernel can hold several at once.
enum ScratchSlot { SCRATCH_COORDS = 0, SCRATCH_CARRY_ROW, SCRATCH_CARRY_VAL, SCRATCH_COUNTER,
                   SCRATCH_STATS, SCRATCH_MISC, SCRATCH_SPMM_X, SCRATCH_SPMM_Y, SCRATCH_XHOT, SCRATCH_NORM,
                   SCRATCH_CG, SCRATCH_ROW_END, SCRATCH_START_MASK, SCRATCH_BICGSTAB, SCRATCH_GMRES,
                   SCRATCH_NUM_SLOTS };
int scratch_get(cudaStream_t stream, ScratchSlot slot, size_t bytes, void **out);

// What the last merge-path partition launched on a (device, stream) wrote, and where: lets a
// caller that vouches for an unchanged matrix (SPMVB200_FLAG_STATIC_PATTERN) skip the search.
struct PartitionTag {
    const void *coords, *Ap;
    int64_t n_rows, nnz, tile_items, n_coords;
    bool operator==(const PartitionTag &o) const {
        return coords == o.coords && Ap == o.Ap && n_rows == o.n_rows && nnz == o.nnz &&
               tile_items == o.tile_items && n_coords == o.n_coords;
    }
};
bool partition_tag_matches(cudaStream_t stream, const PartitionTag &tag);
void partition_tag_store(cudaStream_t stream, const PartitionTag &tag);
// The persistent merge kernel's tile descriptors (merge.cu) are derived from the coordinates of the
// last partition on a (device, stream); a new search makes them stale.  tile_desc_current: the
// descriptors at (row_end, start_mask) were built from those coordinates.
bool tile_desc_current(cudaStream_t stream, const void *row_end, const void *start_mask);
void tile_desc_store(cudaStream_t stream, const void *row_end, const void *start_mask);
void scratch_release_all();

int64_t option_get(const char *name, int64_t fallback);

// Option "side_stream" (default 0): a small kernel that a big one depends on (the merge-path
// partition, the refill of x_hot) is launched on a side stream, forked from and joined to the
// caller's stream with events.  Built against a ~170 us idle gap that the CUPTI timeline
// (tools/step_kernels.py, torch profiler) shows between such a kernel and the tile kernel behind
// it -- and which the fork / join removes *in that timeline*.  Event timing outside the profiler
// shows no such gap (back-to-back R-MAT scale 24 SpMVs: 1121 us without, 1124 us with the side
// stream; power-iteration step 11.13 / 11.16 ms), and the extra streams cost the three-slot
// host-buffer pipeline its overlap (11.7 -> 19.0 ms per step end to end).  A profiler artefact:
// off.  profiles/r2_step_kernels.txt keeps the whole chase.
int side_fork(cudaStream_t stream, cudaStream_t *side);
int side_join(cudaStream_t stream);

// cudaEvent bracket around the dominant kernel of a call (no-op unless "time_main_kernel")
class KernelTimerScope {
public:
    explicit KernelTimerScope(cudaStream_t s);
    ~KernelTimerScope();
    KernelTimerScope(const KernelTimerScope &) = delete;
    KernelTimerScope &operator=(const KernelTimerScope &) = delete;

private:
    cudaStream_t stream_;
    cudaEvent_t a_ = nullptr, b_ = nullptr;
    bool active_ = false;
};
void kernel_timer_read(double *total_ms, int64_t *launches);

// Extra destinations of every y store (peer GPUs' replicas of the next x).
constexpr int kMaxPeers = 8;
struct PeerOut {
    void *ptr[kMaxPeers];
    int n;
};

template <typename OffT, typename ValT>
struct SpmvProblem {
    int32_t n_rows;
    int32_t n_cols;
    OffT nnz;
    const OffT *Ap;
    const int32_t *Aj;
    const ValT *Ax;
    const ValT *x;
    ValT *y;
    const ValT *alpha_dev;  // device scalar or nullptr (= 1)
    PeerOut peers;
    cudaStream_t stream;
    bool reuse_partition = false;  // SPMVB200_FLAG_STATIC_PATTERN: tile coordinates may be reused
};

// launchers (one translation unit each)
template <typename OffT, typename ValT> int launch_merge(const SpmvProblem<OffT, ValT> &p);
template <typename OffT, typename ValT>
int launch_merge_genl(const SpmvProblem<OffT, ValT> &p, int semiring, const ValT *beta_dev);
template <typename OffT, typename ValT> int launch_vector(const SpmvProblem<OffT, ValT> &p, int width);
template <typename OffT, typename ValT> int launch_light(const SpmvProblem<OffT, ValT> &p, int width);
template <typename OffT, typename ValT> int launch_stream(const SpmvProblem<OffT, ValT> &p);
template <typename OffT, typename ValT> int launch_cusparse(const SpmvProblem<OffT, ValT> &p);
template <typename OffT, typename ValT> int launch_auto(const SpmvProblem<OffT, ValT> &p);
template <typename OffT>
int launch_partition(int32_t n_rows, OffT nnz, const OffT *Ap, int64_t tile_items, int64_t n_coords,
                     int32_t *coords_x, cudaStream_t stream, bool reuse = false);
template <typename OffT>
int row_stats(int64_t n_rows, int64_t nnz, const OffT *Ap, spmvb200_row_stats_t *out,
              cudaStream_t stream, bool use_cache);
int pick_width_from_mean(double mean_row_len);
template <typename OffT, typename ValT>
int launch_spmm(int k, int32_t n_rows, int32_t n_cols, OffT nnz, const OffT *Ap, const int32_t *Aj,
                const ValT *Ax, const ValT *X, int64_t ldx, ValT *Y, int64_t ldy, const ValT *alpha_dev,
                cudaStream_t stream);
// conjugate gradients (cg.cu); arguments checked by the caller
template <typename OffT, typename ValT>
int cg_solve(const spmvb200_cg_args_t &a, spmvb200_cg_result_t *out);
// BiCGSTAB (bicgstab.cu); arguments checked by the caller
template <typename OffT, typename ValT>
int bicgstab_solve(const spmvb200_cg_args_t &a, spmvb200_cg_result_t *out);
// restarted GMRES (gmres.cu); arguments, restart included, checked by the caller
template <typename OffT, typename ValT>
int gmres_solve(const spmvb200_cg_args_t &a, int restart, spmvb200_cg_result_t *out);

// The hot part of x, compacted (hotx.cu): a per-matrix plan holding a remapped copy of Aj (hot
// column c stored as 0x80000000 | rank) and the list of hot columns; x_hot lives in the
// per-stream scratch (calls on different streams may share a plan) and is refilled from x by
// hot_gather before every SpMV that uses the plan.
struct HotPlan {
    const int32_t *Aj2 = nullptr;
    const int32_t *hot_cols = nullptr;
    int64_t K = 0;
    int64_t K_table = 0;      // ranks 0 .. K_table-1: the most frequent columns (shared-memory table class)
    int32_t n_cols = 0;
    uint32_t threshold = 0;   // a column is hot when it occurs at least this often
    double hot_share = 0.0;   // fraction of the gathers that go to hot columns
    double table_share = 0.0; // ... and to the table class
    double build_ms = 0.0;
};
int hot_plan_get(const int32_t *Aj, int64_t nnz, int32_t n_cols, int64_t k_max, int64_t k_table, cudaStream_t stream,
                 bool may_build, const HotPlan **out);
template <typename ValT> int hot_gather(const HotPlan &plan, const ValT *x, cudaStream_t stream, const ValT **x_hot);
void hot_plan_clear();
void hot_plan_drop(const int32_t *Aj);
const HotPlan *hot_plan_peek(const int32_t *Aj);  // the plan built for this Aj on the current device, or nullptr

int gather_yardstick(int64_t n_x, int64_t count, int reps, cudaStream_t stream, double *best_ms);

// Launch attribute helper: optional L2 access-policy window over x (option "l2_window").
struct LaunchCfg {
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attrs[2];
};
void make_launch_cfg(LaunchCfg &lc, dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                     const void *x, size_t x_bytes);

#ifdef __CUDACC__
// ------------------------------------------------------------------ device: PTX wrappers

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// make the init visible to the async (TMA) proxy
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}

// L2 eviction policies (createpolicy): streams are read once, x is re-read.
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}

// TMA 1-D bulk copy global -> shared, completion on an mbarrier.  dst, src 16-byte
// aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gsrc, uint32_t bytes,
                                         uint64_t *bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
        "[%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(smem_dst)),
        "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}

// gather of x with an L2 policy (evict_last keeps x resident against the Aj/Ax stream).
// SPMV_GATHER_MODE selects the load flavour at compile time (ablation; default 0):
//   0  ld.global.nc + L2::cache_hint(evict_last)      1  ld.global.cg (bypass L1)
//   2  ld.global.nc.L1::no_allocate + L2 hint         3  plain ld.global.nc
//   4  ld.global.nc.L2::128B (whole line on an L2 miss)   5  4 + evict_last hint
//   6  ld.global.nc.L2::256B                              7  ld.global.nc.L2::64B
#ifndef SPMV_GATHER_MODE
#define SPMV_GATHER_MODE 0
#endif
#if SPMV_GATHER_MODE == 0
#define SPMV_GATHER_ASM(T, C) "ld.global.nc.L2::cache_hint." T " %0, [%1], %2;" : "=" C(v) : "l"(p), "l"(policy)
#elif SPMV_GATHER_MODE == 1
#define SPMV_GATHER_ASM(T, C) "ld.global.cg." T " %0, [%1];" : "=" C(v) : "l"(p)
#elif SPMV_GATHER_MODE == 2
#define SPMV_GATHER_ASM(T, C) "ld.global.nc.L1::no_allocate.L2::cache_hint." T " %0, [%1], %2;" : "=" C(v) : "l"(p), "l"(policy)
#elif SPMV_GATHER_MODE == 3
#define SPMV_GATHER_ASM(T, C) "ld.global.nc." T " %0, [%1];" : "=" C(v) : "l"(p)
#elif SPMV_GATHER_MODE == 4
#define SPMV_GATHER_ASM(T, C) "ld.global.nc.L2::128B." T " %0, [%1];" : "=" C(v) : "l"(p)
#elif SPMV_GATHER_MODE == 5
#define SPMV_GATHER_ASM(T, C) "ld.global.nc.L2::cache_hint.L2::128B." T " %0, [%1], %2;" : "=" C(v) : "l"(p), "l"(policy)
#elif SPMV_GATHER_MODE == 6
#define SPMV_GATHER_ASM(T, C) "ld.global.nc.L2::256B." T " %0, [%1];" : "=" C(v) : "l"(p)
#else
#define SPMV_GATHER_ASM(T, C) "ld.global.nc.L2::64B." T " %0, [%1];" : "=" C(v) : "l"(p)
#endif
__device__ __forceinline__ float ldg_hint(const float *p, uint64_t policy) {
    float v;
    asm volatile(SPMV_GATHER_ASM("f32", "f"));
    return v;
}
__device__ __forceinline__ double ldg_hint(const double *p, uint64_t policy) {
    double v;
    asm volatile(SPMV_GATHER_ASM("f64", "d"));
    return v;
}

// 128-bit streaming loads (read once: no L1 allocation, L2 evict-first policy)
__device__ __forceinline__ int4 ldg_stream_int4(const int32_t *p, uint64_t policy) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.s32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p), "l"(policy));
    return r;
}
__device__ __forceinline__ float4 ldg_stream_val4(const float *p, uint64_t policy) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p), "l"(policy));
    return r;
}
struct double4_t {
    double x, y, z, w;
};
__device__ __forceinline__ double4_t ldg_stream_val4(const double *p, uint64_t policy) {
    double4_t r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.f64 {%0,%1}, [%2], %3;"
                 : "=d"(r.x), "=d"(r.y)
                 : "l"(p), "l"(policy));
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.f64 {%0,%1}, [%2], %3;"
                 : "=d"(r.z), "=d"(r.w)
                 : "l"(p + 2), "l"(policy));
    return r;
}

template <typename ValT> struct Val4;
template <> struct Val4<float> { using type = float4; };
template <> struct Val4<double> { using type = double4_t; };

// sum over the T lanes of a sub-warp (T a power of two <= 32); every lane gets the total
template <int T, typename ValT>
__device__ __forceinline__ ValT subwarp_sum(ValT v) {
#pragma unroll
    for (int s = T / 2; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s, 32);
    return v;
}

// NVLink multicast store (NVLS): one store, the switch replicates it into every GPU bound to
// the multicast object, the storing GPU included.
__device__ __forceinline__ void multimem_st(float *mc, float v) {
    asm volatile("multimem.st.weak.global.f32 [%0], %1;" ::"l"(mc), "f"(v) : "memory");
}
__device__ __forceinline__ void multimem_st(double *mc, double v) {
    asm volatile("multimem.st.weak.global.f64 [%0], %1;" ::"l"(mc), "d"(v) : "memory");
}

// fan a y value out to the replicas of the other GPUs: peers.n > 0 -> that many peer-mapped
// pointers; peers.n == -1 -> ptr[0] is a multicast address covering all replicas
template <typename ValT>
__device__ __forceinline__ void store_peers(const PeerOut &peers, int64_t row, ValT v) {
    if (peers.n < 0) {
        multimem_st(static_cast<ValT *>(peers.ptr[0]) + row, v);
    } else {
#pragma unroll
        for (int i = 0; i < kMaxPeers; ++i)
            if (i < peers.n) static_cast<ValT *>(peers.ptr[i])[row] = v;
    }
}

// y store fanned out to the peer replicas
template <typename ValT>
__device__ __forceinline__ void store_y(ValT *y, const PeerOut &peers, int64_t row, ValT v) {
    y[row] = v;
    store_peers(peers, row, v);
}
// Row stores of the SpMV kernels: the local y always; the peer replicas only when the row has
// nonzeros.  An empty row's y is 0 on every step, and the replicas start out zeroed
// (dist.PowerIteration), so its value never has to cross NVLink.  On R-MAT scale 27, 61 % of
// the rows are empty and the rank owning the sparse tail would otherwise send 7 x 218 MB per
// step -- the fused exchange was egress-bound on that one rank (4.2 ms/step at 8 GPUs against
// a 2.1 ms kernel).  A row whose nonzeros all lie in earlier tiles gets its value from the
// merge fixup, which always stores to the peers.
template <typename ValT>
__device__ __forceinline__ void store_y_nonempty(ValT *y, const PeerOut &peers, int64_t row, ValT v,
                                                 bool has_nonzeros) {
    y[row] = v;
    if (has_nonzeros) store_peers(peers, row, v);
}
#endif  // __CUDACC__

// ---- mcast.cu: device memory replicated over the GPUs of this process behind one NVLink
// multicast address (NVLS).  SPMVB200_ERR_UNSUPPORTED without multicast support.
struct McastArena;
int mcast_arena_create(const int *devices, int n, size_t bytes, McastArena **out, void **replica, void **mc);
void mcast_arena_destroy(McastArena *a);

}  // namespace spmvb200
