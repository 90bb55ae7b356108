// api.cu -- the extern "C" surface declared in include/spmv_b200.h.
//
// Argument checking, type dispatch and the host-buffer convenience object live here; the
// kernels are in merge.cu / vector.cu / light.cu, the selector and cuSPARSE baseline in
// select.cu, the data layer in gen.cu.
#include <cstring>
#include <new>
#include <vector>

#include "common.cuh"

namespace spmvb200 {
int64_t merge_tile_items(int offset_bits);
void stats_cache_clear();
void cusparse_plan_clear();
template <typename ValT>
int gen_uniform_pm1(uint64_t, uint32_t, uint64_t, int64_t, ValT *, cudaStream_t);
template <typename OffT, typename ValT>
int gen_lap2d(int32_t, OffT *, int32_t *, ValT *, cudaStream_t);
template <typename OffT, typename ValT>
int gen_uniform_rows(int32_t, int32_t, int32_t, uint64_t, OffT *, int32_t *, ValT *, cudaStream_t);
int gen_rmat_edges(int32_t, uint64_t, uint64_t, int64_t, int32_t *, int32_t *, cudaStream_t);
template <typename OffT, typename ValT>
int coo_to_csr(int32_t, int64_t, int32_t *, int32_t *, const ValT *, OffT *, int32_t *, ValT *,
               cudaStream_t);

namespace {

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

template <typename OffT, typename ValT>
int run(int kind, int64_t n_rows, int64_t n_cols, int64_t nnz, const void *Ap, const int32_t *Aj,
        const void *Ax, const void *x, void *y, const void *alpha_dev, void *const *y_peers,
        int n_peers, cudaStream_t stream, int semiring = SPMVB200_SEMIRING_PLUS_TIMES,
        const void *beta_dev = nullptr, int flags = 0) {
    if (n_rows < 0 || n_cols < 0 || nnz < 0) return SPMVB200_ERR_INVALID;
    if (n_rows > 0x7fffffffLL || n_cols > 0x7fffffffLL) return SPMVB200_ERR_INVALID;
    if (sizeof(OffT) == 4 && nnz > 0x7fffffffLL) return SPMVB200_ERR_INVALID;
    // 32-bit offset arithmetic steps up to 1024 positions past a row end before it compares
    if (sizeof(OffT) == 4 && nnz > 0x7fffffffLL - 4096) return SPMVB200_ERR_UNSUPPORTED;
    // the reference's no-op case (merge_based/dispatch_spmv_orig.cuh:564-570) is n_rows == 0 or
    // n_cols == 0.  Without rows there is nothing to write; without columns there can be no
    // nonzeros, and "y is fully overwritten" still has to hold: every row is an empty row, so the
    // call goes on like any other (y = identity, or beta * y) -- unless the caller, counting on
    // the no-op, passed no offsets at all, in which case y = 0 is written directly.
    if (n_rows == 0) return SPMVB200_OK;
    if (n_cols == 0) {
        if (nnz != 0) return SPMVB200_ERR_INVALID;
        if (!y) return SPMVB200_ERR_INVALID;
        if (!Ap) {
            if (semiring != SPMVB200_SEMIRING_PLUS_TIMES || beta_dev || n_peers != 0) return SPMVB200_ERR_INVALID;
            SPMV_CUDA_TRY(cudaMemsetAsync(y, 0, (size_t)n_rows * sizeof(ValT), stream));
            return SPMVB200_OK;
        }
    }
    if (!Ap || !y || (nnz > 0 && (!Aj || !Ax || !x))) return SPMVB200_ERR_INVALID;
    if (!aligned16(Ap) || !aligned16(Aj) || !aligned16(Ax)) return SPMVB200_ERR_ALIGNMENT;
    // n_peers == -1: y_peers[0] is an NVLink multicast address (one store reaches every replica)
    if (n_peers < -1 || n_peers > kMaxPeers || (n_peers != 0 && (!y_peers || !y_peers[0]))) return SPMVB200_ERR_INVALID;

    SpmvProblem<OffT, ValT> p;
    p.n_rows = (int32_t)n_rows;
    p.n_cols = (int32_t)n_cols;
    p.nnz = (OffT)nnz;
    p.Ap = static_cast<const OffT *>(Ap);
    p.Aj = Aj;
    p.Ax = static_cast<const ValT *>(Ax);
    p.x = static_cast<const ValT *>(x);
    p.y = static_cast<ValT *>(y);
    p.alpha_dev = static_cast<const ValT *>(alpha_dev);
    p.peers.n = n_peers;
    for (int i = 0; i < kMaxPeers; ++i) p.peers.ptr[i] = i < (n_peers < 0 ? 1 : n_peers) ? y_peers[i] : nullptr;
    p.stream = stream;
    // option "assume_static_pattern": the vouching of SPMVB200_FLAG_STATIC_PATTERN for callers whose
    // call has no flags argument (the reference's SpMV(kind_str, ...) plugin surface)
    p.reuse_partition = (flags & SPMVB200_FLAG_STATIC_PATTERN) != 0 || option_get("assume_static_pattern", 0) != 0;

    if (semiring != SPMVB200_SEMIRING_PLUS_TIMES || beta_dev) {
        // the generalised form lives in the merge-path kernel only (as in the reference)
        if (kind != SPMVB200_KIND_MERGE && kind != SPMVB200_KIND_AUTO) return SPMVB200_ERR_UNSUPPORTED;
        return launch_merge_genl<OffT, ValT>(p, semiring, static_cast<const ValT *>(beta_dev));
    }
    switch (kind) {
        case SPMVB200_KIND_MERGE: return launch_merge<OffT, ValT>(p);
        case SPMVB200_KIND_VECTOR: return launch_vector<OffT, ValT>(p, 0);
        case SPMVB200_KIND_LIGHT: return launch_light<OffT, ValT>(p, 0);
        case SPMVB200_KIND_STREAM: return launch_stream<OffT, ValT>(p);
        case SPMVB200_KIND_AUTO: return launch_auto<OffT, ValT>(p);
        case SPMVB200_KIND_CUSPARSE: return launch_cusparse<OffT, ValT>(p);
        default: return SPMVB200_ERR_INVALID;
    }
}

int run_untyped(const spmvb200_args_t *a) {
    if (!a) return SPMVB200_ERR_INVALID;
    if (a->flags & ~SPMVB200_FLAG_STATIC_PATTERN) return SPMVB200_ERR_INVALID;
    cudaStream_t s = static_cast<cudaStream_t>(a->stream);
#define GO(O, V)                                                                              \
    return run<O, V>(a->kind, a->n_rows, a->n_cols, a->nnz, a->Ap, a->Aj, a->Ax, a->x, a->y,  \
                     a->alpha_dev, a->y_peers, a->n_peers, s, a->semiring, a->beta_dev, a->flags)
    if (a->offset_bits == 32 && a->value_bits == 32) GO(int32_t, float);
    if (a->offset_bits == 32 && a->value_bits == 64) GO(int32_t, double);
    if (a->offset_bits == 64 && a->value_bits == 32) GO(int64_t, float);
    if (a->offset_bits == 64 && a->value_bits == 64) GO(int64_t, double);
#undef GO
    return SPMVB200_ERR_UNSUPPORTED;
}

}  // namespace
}  // namespace spmvb200

using namespace spmvb200;

extern "C" {

// ---- typed hot-path symbols ---------------------------------------------------------------
#define SPMVB200_DEFINE(KIND, KIND_ENUM, OTAG, OFF_T, VTAG, VAL_T)                              \
    int spmvb200_##KIND##_i32_##OTAG##_##VTAG(int32_t n_rows, int32_t n_cols, OFF_T nnz,        \
                                              const OFF_T *Ap, const int32_t *Aj,               \
                                              const VAL_T *Ax, const VAL_T *x, VAL_T *y,        \
                                              spmvb200_stream_t stream) {                       \
        return run<OFF_T, VAL_T>(KIND_ENUM, n_rows, n_cols, (int64_t)nnz, Ap, Aj, Ax, x, y,     \
                                 nullptr, nullptr, 0, static_cast<cudaStream_t>(stream));       \
    }
#define SPMVB200_DEFINE_KIND(KIND, KIND_ENUM)                       \
    SPMVB200_DEFINE(KIND, KIND_ENUM, o32, int32_t, f32, float)      \
    SPMVB200_DEFINE(KIND, KIND_ENUM, o32, int32_t, f64, double)     \
    SPMVB200_DEFINE(KIND, KIND_ENUM, o64, int64_t, f32, float)      \
    SPMVB200_DEFINE(KIND, KIND_ENUM, o64, int64_t, f64, double)
SPMVB200_DEFINE_KIND(merge, SPMVB200_KIND_MERGE)
SPMVB200_DEFINE_KIND(vector, SPMVB200_KIND_VECTOR)
SPMVB200_DEFINE_KIND(light, SPMVB200_KIND_LIGHT)
SPMVB200_DEFINE_KIND(stream, SPMVB200_KIND_STREAM)
SPMVB200_DEFINE_KIND(auto, SPMVB200_KIND_AUTO)
SPMVB200_DEFINE_KIND(cusparse, SPMVB200_KIND_CUSPARSE)

int spmvb200_spmv(const spmvb200_args_t *args) { return run_untyped(args); }

int spmvb200_spmm(const spmvb200_spmm_args_t *a) {
    if (!a || a->n_rows < 0 || a->n_cols < 0 || a->nnz < 0) return SPMVB200_ERR_INVALID;
    if (a->n_rows > 0x7fffffffLL || a->n_cols > 0x7fffffffLL) return SPMVB200_ERR_INVALID;
    if (a->k != 2 && a->k != 4 && a->k != 8) return SPMVB200_ERR_UNSUPPORTED;
    if (a->n_rows == 0 || a->n_cols == 0) return SPMVB200_OK;
    if (!a->Ap || !a->Y || (a->nnz > 0 && (!a->Aj || !a->Ax || !a->X))) return SPMVB200_ERR_INVALID;
    if (a->ldx < a->k || a->ldy < a->k) return SPMVB200_ERR_INVALID;
    if (a->offset_bits == 32 && a->nnz > 0x7fffffffLL - 4096) return SPMVB200_ERR_UNSUPPORTED;
    if (!aligned16(a->Ap) || !aligned16(a->Aj) || !aligned16(a->Ax)) return SPMVB200_ERR_ALIGNMENT;
    const size_t vb = a->value_bits / 8;
    const size_t row_align = (size_t)a->k * vb >= 16 ? 16 : 8;
    auto ok = [&](const void *p, int64_t ld) {
        return (reinterpret_cast<uintptr_t>(p) % row_align) == 0 && ((size_t)ld * vb) % row_align == 0;
    };
    if (!ok(a->X, a->ldx) || !ok(a->Y, a->ldy)) return SPMVB200_ERR_ALIGNMENT;
    cudaStream_t s = static_cast<cudaStream_t>(a->stream);
#define GO(O, V)                                                                                      \
    return launch_spmm<O, V>(a->k, (int32_t)a->n_rows, (int32_t)a->n_cols, (O)a->nnz,                  \
                             static_cast<const O *>(a->Ap), a->Aj, static_cast<const V *>(a->Ax),      \
                             static_cast<const V *>(a->X), a->ldx, static_cast<V *>(a->Y), a->ldy,     \
                             static_cast<const V *>(a->alpha_dev), s)
    if (a->offset_bits == 32 && a->value_bits == 32) GO(int32_t, float);
    if (a->offset_bits == 32 && a->value_bits == 64) GO(int32_t, double);
    if (a->offset_bits == 64 && a->value_bits == 32) GO(int64_t, float);
    if (a->offset_bits == 64 && a->value_bits == 64) GO(int64_t, double);
#undef GO
    return SPMVB200_ERR_UNSUPPORTED;
}

// ---- Krylov solvers: conjugate gradients, BiCGSTAB, GMRES -----------------------------------
// Every argument is checked here, before any CUDA call (so also without a device); then
// solve(OffT(), ValT()) runs the solver for the offset and value widths.
extern "C++" {
template <typename Solve>
static int krylov_entry(const spmvb200_cg_args_t *a, spmvb200_cg_result_t *out, Solve solve) {
    if (!a || !out) return SPMVB200_ERR_INVALID;
    if (a->kind < SPMVB200_KIND_MERGE || a->kind > SPMVB200_KIND_STREAM) return SPMVB200_ERR_INVALID;
    if (a->flags & ~SPMVB200_CG_JACOBI) return SPMVB200_ERR_INVALID;
    if (!(a->rtol > 0.0) || a->max_iter < 0 || a->n < 0 || a->nnz < 0) return SPMVB200_ERR_INVALID;
    if ((a->offset_bits != 32 && a->offset_bits != 64) || (a->value_bits != 32 && a->value_bits != 64))
        return SPMVB200_ERR_UNSUPPORTED;
    if (a->n > 0x7fffffffLL) return SPMVB200_ERR_INVALID;
    if (a->offset_bits == 32 && a->nnz > 0x7fffffffLL - 4096) return SPMVB200_ERR_UNSUPPORTED;
    if (a->n == 0) {
        std::memset(out, 0, sizeof(*out));
        out->converged = 1;
        return SPMVB200_OK;
    }
    if (!a->Ap || !a->b || !a->x || (a->nnz > 0 && (!a->Aj || !a->Ax))) return SPMVB200_ERR_INVALID;
    if (a->x == a->b) return SPMVB200_ERR_INVALID;
    if (!aligned16(a->Ap) || !aligned16(a->Aj) || !aligned16(a->Ax)) return SPMVB200_ERR_ALIGNMENT;
    if (a->offset_bits == 32) return a->value_bits == 32 ? solve(int32_t(), float()) : solve(int32_t(), double());
    return a->value_bits == 32 ? solve(int64_t(), float()) : solve(int64_t(), double());
}
}

int spmvb200_cg(const spmvb200_cg_args_t *a, spmvb200_cg_result_t *out) {
    return krylov_entry(a, out, [&](auto o, auto v) { return cg_solve<decltype(o), decltype(v)>(*a, out); });
}

int spmvb200_bicgstab(const spmvb200_cg_args_t *a, spmvb200_cg_result_t *out) {
    return krylov_entry(a, out, [&](auto o, auto v) { return bicgstab_solve<decltype(o), decltype(v)>(*a, out); });
}

int spmvb200_gmres(const spmvb200_cg_args_t *a, int32_t restart, spmvb200_cg_result_t *out) {
    if (restart < 1 || restart > SPMVB200_GMRES_MAX_RESTART) return SPMVB200_ERR_INVALID;
    return krylov_entry(a, out,
                        [&](auto o, auto v) { return gmres_solve<decltype(o), decltype(v)>(*a, restart, out); });
}

// ---- partition / row split -----------------------------------------------------------------
int spmvb200_merge_path_partition_o32(int32_t n_rows, int32_t nnz, const int32_t *Ap,
                                      int64_t tile_items, int64_t n_coords, int32_t *coords_x,
                                      spmvb200_stream_t stream) {
    if (n_rows < 0 || nnz < 0 || tile_items <= 0 || n_coords < 0 || !Ap || !coords_x)
        return SPMVB200_ERR_INVALID;
    return launch_partition<int32_t>(n_rows, nnz, Ap, tile_items, n_coords, coords_x,
                                     static_cast<cudaStream_t>(stream));
}
int spmvb200_merge_path_partition_o64(int32_t n_rows, int64_t nnz, const int64_t *Ap,
                                      int64_t tile_items, int64_t n_coords, int32_t *coords_x,
                                      spmvb200_stream_t stream) {
    if (n_rows < 0 || nnz < 0 || tile_items <= 0 || n_coords < 0 || !Ap || !coords_x)
        return SPMVB200_ERR_INVALID;
    return launch_partition<int64_t>(n_rows, nnz, Ap, tile_items, n_coords, coords_x,
                                     static_cast<cudaStream_t>(stream));
}
int64_t spmvb200_merge_tile_items(int offset_bits, int) { return merge_tile_items(offset_bits); }

}  // extern "C"

namespace spmvb200 {
// Weighted variant of the same search: the cost of the first r rows is
// f(r) = w_den * Ap[r] + w_num * r (a row costs w_num / w_den of a nonzero; 1/1 is the merge
// path), and out[k] = max{ r in [0, n_rows] : f(r) <= targets[k] }.  One thread per target.
template <typename OffT>
__global__ void rows_at_cost_kernel(int32_t n_rows, const OffT *__restrict__ Ap, int64_t w_num,
                                    int64_t w_den, int n_targets, const int64_t *__restrict__ targets,
                                    int64_t *__restrict__ rows_out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_targets) return;
    const int64_t d = targets[k];
    int64_t lo = 0, hi = n_rows;  // f(0) = 0 <= d for every d >= 0
    while (lo < hi) {
        const int64_t mid = lo + ((hi - lo + 1) >> 1);
        const int64_t f = w_den * (int64_t)__ldg(Ap + mid) + w_num * mid;
        if (f <= d) lo = mid; else hi = mid - 1;
    }
    rows_out[k] = lo;
}
}  // namespace spmvb200

namespace {
// diagonals floor(g*total/parts) are not an arithmetic progression in general, so the split
// reuses the partition kernel once per boundary with tile_items = that diagonal, n_coords = 2
// (coordinate 1 is the one wanted).  parts is tiny.
template <typename OffT>
int row_split_impl(int32_t n_rows, OffT nnz, const OffT *Ap, int parts, int64_t *row_bounds,
                   cudaStream_t stream) {
    if (parts < 1 || !row_bounds || n_rows < 0 || nnz < 0 || (!Ap && n_rows > 0))
        return SPMVB200_ERR_INVALID;
    const int64_t total = (int64_t)n_rows + (int64_t)nnz;
    void *dbuf = nullptr;
    SPMV_TRY(scratch_get(stream, SCRATCH_MISC, (size_t)(parts + 1) * 2 * sizeof(int32_t), &dbuf));
    int32_t *d = static_cast<int32_t *>(dbuf);
    row_bounds[0] = 0;
    for (int g = 1; g < parts; ++g) {
        const int64_t diag = (int64_t)(((__int128)g * (__int128)total) / parts);
        if (diag == 0) {
            SPMV_CUDA_TRY(cudaMemsetAsync(d + 2 * g, 0, 2 * sizeof(int32_t), stream));
        } else {
            SPMV_TRY(launch_partition<OffT>(n_rows, nnz, Ap, diag, 2, d + 2 * g, stream));
        }
    }
    std::vector<int32_t> h((size_t)(parts + 1) * 2, 0);
    if (parts > 1)
        SPMV_CUDA_TRY(cudaMemcpyAsync(h.data(), d, h.size() * sizeof(int32_t), cudaMemcpyDeviceToHost,
                                      stream));
    SPMV_CUDA_TRY(cudaStreamSynchronize(stream));
    for (int g = 1; g < parts; ++g) row_bounds[g] = h[2 * g + 1];
    row_bounds[parts] = n_rows;
    return SPMVB200_OK;
}

template <typename OffT>
int rows_at_cost_impl(int32_t n_rows, const OffT *Ap, int64_t w_num, int64_t w_den, int n_targets,
                      const int64_t *targets, int64_t *rows_out, cudaStream_t stream) {
    if (n_rows < 0 || (!Ap && n_rows > 0) || w_num < 0 || w_den < 1 || n_targets < 0 ||
        (n_targets > 0 && (!targets || !rows_out)))
        return SPMVB200_ERR_INVALID;
    // f must stay inside int64: Ap[r] < 2^63 / (2 * w_den) is implied by these bounds
    if (w_num > (1 << 20) || w_den > (1 << 20)) return SPMVB200_ERR_UNSUPPORTED;
    if (n_targets == 0) return SPMVB200_OK;
    for (int k = 0; k < n_targets; ++k)
        if (targets[k] < 0) return SPMVB200_ERR_INVALID;
    if (n_rows == 0) {
        for (int k = 0; k < n_targets; ++k) rows_out[k] = 0;
        return SPMVB200_OK;
    }
    void *dbuf = nullptr;
    SPMV_TRY(scratch_get(stream, SCRATCH_MISC, (size_t)n_targets * 2 * sizeof(int64_t), &dbuf));
    int64_t *d_t = static_cast<int64_t *>(dbuf), *d_r = d_t + n_targets;
    SPMV_CUDA_TRY(cudaMemcpyAsync(d_t, targets, (size_t)n_targets * sizeof(int64_t), cudaMemcpyHostToDevice,
                                  stream));
    spmvb200::rows_at_cost_kernel<OffT><<<(n_targets + 127) / 128, 128, 0, stream>>>(n_rows, Ap, w_num, w_den,
                                                                           n_targets, d_t, d_r);
    SPMV_LAUNCH_CHECK();
    SPMV_CUDA_TRY(cudaMemcpyAsync(rows_out, d_r, (size_t)n_targets * sizeof(int64_t), cudaMemcpyDeviceToHost,
                                  stream));
    SPMV_CUDA_TRY(cudaStreamSynchronize(stream));
    return SPMVB200_OK;
}
}  // namespace

extern "C" {

int spmvb200_rows_at_cost_o32(int32_t n_rows, const int32_t *Ap, int64_t w_num, int64_t w_den,
                              int n_targets, const int64_t *targets, int64_t *rows_out,
                              spmvb200_stream_t stream) {
    return rows_at_cost_impl<int32_t>(n_rows, Ap, w_num, w_den, n_targets, targets, rows_out,
                                      static_cast<cudaStream_t>(stream));
}
int spmvb200_rows_at_cost_o64(int32_t n_rows, const int64_t *Ap, int64_t w_num, int64_t w_den,
                              int n_targets, const int64_t *targets, int64_t *rows_out,
                              spmvb200_stream_t stream) {
    return rows_at_cost_impl<int64_t>(n_rows, Ap, w_num, w_den, n_targets, targets, rows_out,
                                      static_cast<cudaStream_t>(stream));
}

int spmvb200_row_split_o32(int32_t n_rows, int32_t nnz, const int32_t *Ap, int parts,
                           int64_t *row_bounds, spmvb200_stream_t stream) {
    return row_split_impl<int32_t>(n_rows, nnz, Ap, parts, row_bounds, static_cast<cudaStream_t>(stream));
}
int spmvb200_row_split_o64(int32_t n_rows, int64_t nnz, const int64_t *Ap, int parts,
                           int64_t *row_bounds, spmvb200_stream_t stream) {
    return row_split_impl<int64_t>(n_rows, nnz, Ap, parts, row_bounds, static_cast<cudaStream_t>(stream));
}

// ---- statistics ----------------------------------------------------------------------------
int spmvb200_row_stats(int offset_bits, int64_t n_rows, int64_t nnz, const void *Ap,
                       spmvb200_row_stats_t *out, spmvb200_stream_t stream) {
    if (!out || n_rows < 0 || nnz < 0 || (!Ap && n_rows > 0)) return SPMVB200_ERR_INVALID;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (offset_bits == 32) return row_stats<int32_t>(n_rows, nnz, static_cast<const int32_t *>(Ap), out, s, false);
    if (offset_bits == 64) return row_stats<int64_t>(n_rows, nnz, static_cast<const int64_t *>(Ap), out, s, false);
    return SPMVB200_ERR_UNSUPPORTED;
}

void spmvb200_release_cache(void) {
    stats_cache_clear();
    cusparse_plan_clear();
    hot_plan_clear();
    scratch_release_all();
}

int spmvb200_gather_yardstick(int64_t x_elements, int64_t gathers, int reps, spmvb200_stream_t stream,
                              double *best_ms) {
    return gather_yardstick(x_elements, gathers, reps, static_cast<cudaStream_t>(stream), best_ms);
}

int spmvb200_hot_x_info(const int32_t *Aj, int64_t *hot_columns, double *hot_share, double *build_ms) {
    // never builds: nnz / n_cols are not needed to look a plan up, so find it by address alone
    if (hot_columns) *hot_columns = 0;
    if (hot_share) *hot_share = 0.0;
    if (build_ms) *build_ms = 0.0;
    const HotPlan *plan = hot_plan_peek(Aj);
    if (plan) {
        if (hot_columns) *hot_columns = plan->K;
        if (hot_share) *hot_share = plan->hot_share;
        if (build_ms) *build_ms = plan->build_ms;
    }
    return SPMVB200_OK;
}

int spmvb200_hot_x_table_info(const int32_t *Aj, int64_t *table_columns, double *table_share) {
    if (table_columns) *table_columns = 0;
    if (table_share) *table_share = 0.0;
    if (const HotPlan *plan = hot_plan_peek(Aj)) {
        if (table_columns) *table_columns = plan->K_table;
        if (table_share) *table_share = plan->table_share;
    }
    return SPMVB200_OK;
}

}  // extern "C"

// ---- host-buffer matrix object -------------------------------------------------------------
struct spmvb200_matrix {
    int offset_bits, value_bits;
    int64_t n_rows, n_cols, nnz;
    void *Ap = nullptr, *Ax = nullptr;
    int32_t *Aj = nullptr;
    bool owns_csr = true;
    // pipeline slots: each has its own stream and device x/y; slot 0 exists from creation, the
    // others are created on first use
    void *x[SPMVB200_MAX_SLOTS] = {}, *y[SPMVB200_MAX_SLOTS] = {};
    cudaStream_t stream[SPMVB200_MAX_SLOTS] = {};
    int64_t calls = 0;
};

namespace spmvb200 {
template <typename ValT> int sum_squares(int64_t, const ValT *, double *, cudaStream_t);
template <typename ValT> int inv_sqrt(const double *, ValT *, cudaStream_t);
template <typename ValT>
int norm_exchange(int64_t, const ValT *, int, int, uint64_t, double *, void *const *, void *, double *, ValT *,
                  int *, cudaStream_t);
}  // namespace spmvb200

extern "C" {

int spmvb200_sum_squares(int value_bits, int64_t n, const void *v, double *sumsq_dev,
                         spmvb200_stream_t stream) {
    if (n < 0 || !sumsq_dev || (n > 0 && !v)) return SPMVB200_ERR_INVALID;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (value_bits == 32) return sum_squares<float>(n, static_cast<const float *>(v), sumsq_dev, s);
    if (value_bits == 64) return sum_squares<double>(n, static_cast<const double *>(v), sumsq_dev, s);
    return SPMVB200_ERR_UNSUPPORTED;
}
int spmvb200_norm_exchange(int value_bits, int64_t n, const void *y_local, int rank, int world,
                           uint64_t step, void *mailbox_local, void *const *mailbox_of_rank,
                           void *mailbox_multicast, double *sumsq_dev, void *alpha_dev, int *error_dev,
                           spmvb200_stream_t stream) {
    if (n < 0 || (n > 0 && !y_local)) return SPMVB200_ERR_INVALID;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (value_bits == 32)
        return norm_exchange<float>(n, static_cast<const float *>(y_local), rank, world, step,
                                    static_cast<double *>(mailbox_local), mailbox_of_rank, mailbox_multicast,
                                    sumsq_dev, static_cast<float *>(alpha_dev), error_dev, s);
    if (value_bits == 64)
        return norm_exchange<double>(n, static_cast<const double *>(y_local), rank, world, step,
                                     static_cast<double *>(mailbox_local), mailbox_of_rank, mailbox_multicast,
                                     sumsq_dev, static_cast<double *>(alpha_dev), error_dev, s);
    return SPMVB200_ERR_UNSUPPORTED;
}

int spmvb200_inv_sqrt(int value_bits, const double *sumsq_dev, void *alpha_dev, spmvb200_stream_t stream) {
    if (!sumsq_dev || !alpha_dev) return SPMVB200_ERR_INVALID;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (value_bits == 32) return inv_sqrt<float>(sumsq_dev, static_cast<float *>(alpha_dev), s);
    if (value_bits == 64) return inv_sqrt<double>(sumsq_dev, static_cast<double *>(alpha_dev), s);
    return SPMVB200_ERR_UNSUPPORTED;
}
int spmvb200_main_kernel_time(double *total_ms, int64_t *launches) {
    if (!total_ms || !launches) return SPMVB200_ERR_INVALID;
    kernel_timer_read(total_ms, launches);
    return SPMVB200_OK;
}
int spmvb200_device_malloc(size_t bytes, void **dev_ptr) {
    if (!dev_ptr) return SPMVB200_ERR_INVALID;
    SPMV_CUDA_TRY(cudaMalloc(dev_ptr, bytes ? bytes : 16));
    return SPMVB200_OK;
}
int spmvb200_device_free(void *dev_ptr) {
    if (dev_ptr) SPMV_CUDA_TRY(cudaFree(dev_ptr));
    return SPMVB200_OK;
}
int spmvb200_matrix_create_from_device(int offset_bits, int value_bits, int64_t n_rows, int64_t n_cols,
                                       int64_t nnz, const void *Ap_dev, const int32_t *Aj_dev,
                                       const void *Ax_dev, spmvb200_matrix_t **out) {
    if (!out || n_rows < 0 || n_cols < 0 || nnz < 0) return SPMVB200_ERR_INVALID;
    if ((offset_bits != 32 && offset_bits != 64) || (value_bits != 32 && value_bits != 64))
        return SPMVB200_ERR_UNSUPPORTED;
    if (!Ap_dev || (nnz > 0 && (!Aj_dev || !Ax_dev))) return SPMVB200_ERR_INVALID;
    spmvb200_matrix *m = new (std::nothrow) spmvb200_matrix;
    if (!m) return SPMVB200_ERR_INVALID;
    m->offset_bits = offset_bits;
    m->value_bits = value_bits;
    m->n_rows = n_rows;
    m->n_cols = n_cols;
    m->nnz = nnz;
    m->owns_csr = false;
    m->Ap = const_cast<void *>(Ap_dev);
    m->Aj = const_cast<int32_t *>(Aj_dev);
    m->Ax = const_cast<void *>(Ax_dev);
    const size_t vb = value_bits / 8;
    cudaError_t e;
    if ((e = cudaStreamCreateWithFlags(&m->stream[0], cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaMalloc(&m->x[0], (size_t)(n_cols ? n_cols : 1) * vb)) != cudaSuccess ||
        (e = cudaMalloc(&m->y[0], (size_t)(n_rows ? n_rows : 1) * vb)) != cudaSuccess) {
        record_cuda_error(e, "matrix_create_from_device", __FILE__, __LINE__);
        spmvb200_matrix_destroy(m);
        return SPMVB200_ERR_CUDA;
    }
    *out = m;
    return SPMVB200_OK;
}

}  // extern "C"

extern "C" {

int spmvb200_matrix_create(int offset_bits, int value_bits, int64_t n_rows, int64_t n_cols,
                           int64_t nnz, const void *Ap_host, const int32_t *Aj_host,
                           const void *Ax_host, spmvb200_matrix_t **out) {
    if (!out || n_rows < 0 || n_cols < 0 || nnz < 0) return SPMVB200_ERR_INVALID;
    if ((offset_bits != 32 && offset_bits != 64) || (value_bits != 32 && value_bits != 64))
        return SPMVB200_ERR_UNSUPPORTED;
    if (!Ap_host || (nnz > 0 && (!Aj_host || !Ax_host))) return SPMVB200_ERR_INVALID;
    spmvb200_matrix *m = new (std::nothrow) spmvb200_matrix;
    if (!m) return SPMVB200_ERR_INVALID;
    m->offset_bits = offset_bits;
    m->value_bits = value_bits;
    m->n_rows = n_rows;
    m->n_cols = n_cols;
    m->nnz = nnz;
    const size_t ob = offset_bits / 8, vb = value_bits / 8;
    auto fail = [&](cudaError_t e, const char *what) {
        record_cuda_error(e, what, __FILE__, __LINE__);
        spmvb200_matrix_destroy(m);
        return SPMVB200_ERR_CUDA;
    };
    cudaError_t e;
    if ((e = cudaStreamCreateWithFlags(&m->stream[0], cudaStreamNonBlocking)) != cudaSuccess) return fail(e, "cudaStreamCreate");
    if ((e = cudaMalloc(&m->Ap, (size_t)(n_rows + 1) * ob)) != cudaSuccess) return fail(e, "cudaMalloc Ap");
    if ((e = cudaMalloc((void **)&m->Aj, (size_t)(nnz ? nnz : 1) * 4)) != cudaSuccess) return fail(e, "cudaMalloc Aj");
    if ((e = cudaMalloc(&m->Ax, (size_t)(nnz ? nnz : 1) * vb)) != cudaSuccess) return fail(e, "cudaMalloc Ax");
    if ((e = cudaMalloc(&m->x[0], (size_t)(n_cols ? n_cols : 1) * vb)) != cudaSuccess) return fail(e, "cudaMalloc x");
    if ((e = cudaMalloc(&m->y[0], (size_t)(n_rows ? n_rows : 1) * vb)) != cudaSuccess) return fail(e, "cudaMalloc y");
    if ((e = cudaMemcpyAsync(m->Ap, Ap_host, (size_t)(n_rows + 1) * ob, cudaMemcpyHostToDevice, m->stream[0])) != cudaSuccess) return fail(e, "H2D Ap");
    if (nnz > 0) {
        if ((e = cudaMemcpyAsync(m->Aj, Aj_host, (size_t)nnz * 4, cudaMemcpyHostToDevice, m->stream[0])) != cudaSuccess) return fail(e, "H2D Aj");
        if ((e = cudaMemcpyAsync(m->Ax, Ax_host, (size_t)nnz * vb, cudaMemcpyHostToDevice, m->stream[0])) != cudaSuccess) return fail(e, "H2D Ax");
    }
    if ((e = cudaStreamSynchronize(m->stream[0])) != cudaSuccess) return fail(e, "sync");
    *out = m;
    return SPMVB200_OK;
}

int spmvb200_matrix_submit_host(spmvb200_matrix_t *m, int kind, int slot, const void *x_host,
                                void *y_host) {
    if (!m || slot < 0 || slot >= SPMVB200_MAX_SLOTS || (!x_host && m->n_cols > 0) ||
        (!y_host && m->n_rows > 0))
        return SPMVB200_ERR_INVALID;
    const size_t vb = m->value_bits / 8;
    if (!m->stream[slot]) SPMV_CUDA_TRY(cudaStreamCreateWithFlags(&m->stream[slot], cudaStreamNonBlocking));
    if (!m->x[slot]) SPMV_CUDA_TRY(cudaMalloc(&m->x[slot], (size_t)(m->n_cols ? m->n_cols : 1) * vb));
    if (!m->y[slot]) SPMV_CUDA_TRY(cudaMalloc(&m->y[slot], (size_t)(m->n_rows ? m->n_rows : 1) * vb));
    cudaStream_t st = m->stream[slot];
    void *dx = m->x[slot], *dy = m->y[slot];
    if (m->n_cols > 0)
        SPMV_CUDA_TRY(cudaMemcpyAsync(dx, x_host, (size_t)m->n_cols * vb, cudaMemcpyHostToDevice, st));
    spmvb200_args_t a;
    std::memset(&a, 0, sizeof(a));
    a.kind = kind;
    a.offset_bits = m->offset_bits;
    a.value_bits = m->value_bits;
    a.n_rows = m->n_rows;
    a.n_cols = m->n_cols;
    a.nnz = m->nnz;
    a.Ap = m->Ap;
    a.Aj = m->Aj;
    a.Ax = m->Ax;
    a.x = dx;
    a.y = dy;
    a.stream = st;
    // the object's CSR arrays are resident and never change: every call after the first may reuse
    // what earlier calls derived from them (tile coordinates per stream, the hot-x plan)
    a.flags = m->calls++ > 0 ? SPMVB200_FLAG_STATIC_PATTERN : 0;
    SPMV_TRY(spmvb200_spmv(&a));
    if (m->n_rows > 0) {
        if (m->n_cols == 0) SPMV_CUDA_TRY(cudaMemsetAsync(dy, 0, (size_t)m->n_rows * vb, st));
        SPMV_CUDA_TRY(cudaMemcpyAsync(y_host, dy, (size_t)m->n_rows * vb, cudaMemcpyDeviceToHost, st));
    }
    return SPMVB200_OK;
}

int spmvb200_matrix_wait(spmvb200_matrix_t *m, int slot) {
    if (!m || slot < 0 || slot >= SPMVB200_MAX_SLOTS) return SPMVB200_ERR_INVALID;
    if (m->stream[slot]) SPMV_CUDA_TRY(cudaStreamSynchronize(m->stream[slot]));
    return SPMVB200_OK;
}

int spmvb200_matrix_spmv_host(spmvb200_matrix_t *m, int kind, const void *x_host, void *y_host) {
    SPMV_TRY(spmvb200_matrix_submit_host(m, kind, 0, x_host, y_host));
    return spmvb200_matrix_wait(m, 0);
}

void spmvb200_matrix_destroy(spmvb200_matrix_t *m) {
    if (!m) return;
    for (cudaStream_t st : m->stream)
        if (st) cudaStreamSynchronize(st);
    if (m->Aj) hot_plan_drop(m->Aj);  // the plan's key is an address about to be reused
    if (m->owns_csr) {
        if (m->Ap) cudaFree(m->Ap);
        if (m->Aj) cudaFree(m->Aj);
        if (m->Ax) cudaFree(m->Ax);
    }
    for (int k = 0; k < SPMVB200_MAX_SLOTS; ++k) {
        if (m->x[k]) cudaFree(m->x[k]);
        if (m->y[k]) cudaFree(m->y[k]);
        if (m->stream[k]) cudaStreamDestroy(m->stream[k]);
    }
    delete m;
}

// ---- generators / data layer ---------------------------------------------------------------
int spmvb200_gen_uniform_pm1(int value_bits, uint64_t seed, uint32_t stream_id, uint64_t first,
                             int64_t count, void *out, spmvb200_stream_t stream) {
    if (count < 0 || (!out && count > 0)) return SPMVB200_ERR_INVALID;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (value_bits == 32) return gen_uniform_pm1<float>(seed, stream_id, first, count, static_cast<float *>(out), s);
    if (value_bits == 64) return gen_uniform_pm1<double>(seed, stream_id, first, count, static_cast<double *>(out), s);
    return SPMVB200_ERR_UNSUPPORTED;
}

#define DISPATCH_OV(FN, ...)                                                                   \
    do {                                                                                       \
        if (offset_bits == 32 && value_bits == 32) return FN<int32_t, float>(__VA_ARGS__);     \
        if (offset_bits == 32 && value_bits == 64) return FN<int32_t, double>(__VA_ARGS__);    \
        if (offset_bits == 64 && value_bits == 32) return FN<int64_t, float>(__VA_ARGS__);     \
        if (offset_bits == 64 && value_bits == 64) return FN<int64_t, double>(__VA_ARGS__);    \
        return SPMVB200_ERR_UNSUPPORTED;                                                       \
    } while (0)

}  // extern "C"

namespace {
template <typename OffT, typename ValT>
int lap2d_v(int32_t n, void *Ap, int32_t *Aj, void *Ax, cudaStream_t s) {
    return gen_lap2d<OffT, ValT>(n, static_cast<OffT *>(Ap), Aj, static_cast<ValT *>(Ax), s);
}
template <typename OffT, typename ValT>
int uniform_rows_v(int32_t n_rows, int32_t n_cols, int32_t K, uint64_t seed, void *Ap, int32_t *Aj,
                   void *Ax, cudaStream_t s) {
    return gen_uniform_rows<OffT, ValT>(n_rows, n_cols, K, seed, static_cast<OffT *>(Ap), Aj,
                                        static_cast<ValT *>(Ax), s);
}
template <typename OffT, typename ValT>
int coo_to_csr_v(int32_t n_rows, int64_t nnz, int32_t *rows, int32_t *cols, const void *vals,
                 void *Ap, int32_t *Aj, void *Ax, cudaStream_t s) {
    return coo_to_csr<OffT, ValT>(n_rows, nnz, rows, cols, static_cast<const ValT *>(vals),
                                  static_cast<OffT *>(Ap), Aj, static_cast<ValT *>(Ax), s);
}
}  // namespace

extern "C" {

int spmvb200_gen_lap2d(int offset_bits, int value_bits, int32_t grid_n, void *Ap, int32_t *Aj,
                       void *Ax, spmvb200_stream_t stream) {
    if (!Ap || !Aj || !Ax) return SPMVB200_ERR_INVALID;
    DISPATCH_OV(lap2d_v, grid_n, Ap, Aj, Ax, static_cast<cudaStream_t>(stream));
}
int spmvb200_gen_uniform_rows(int offset_bits, int value_bits, int32_t n_rows, int32_t n_cols,
                              int32_t row_len, uint64_t seed, void *Ap, int32_t *Aj, void *Ax,
                              spmvb200_stream_t stream) {
    if (!Ap || !Aj || !Ax) return SPMVB200_ERR_INVALID;
    DISPATCH_OV(uniform_rows_v, n_rows, n_cols, row_len, seed, Ap, Aj, Ax, static_cast<cudaStream_t>(stream));
}
int spmvb200_gen_rmat_edges(int32_t scale, uint64_t seed, uint64_t first_edge, int64_t count,
                            int32_t *rows, int32_t *cols, spmvb200_stream_t stream) {
    if (count < 0 || (count > 0 && (!rows || !cols))) return SPMVB200_ERR_INVALID;
    return gen_rmat_edges(scale, seed, first_edge, count, rows, cols, static_cast<cudaStream_t>(stream));
}
int spmvb200_coo_to_csr(int offset_bits, int value_bits, int32_t n_rows, int64_t nnz, int32_t *rows,
                        int32_t *cols, const void *vals, void *Ap, int32_t *Aj, void *Ax,
                        spmvb200_stream_t stream) {
    if (!Ap || (nnz > 0 && (!rows || !cols || !Aj)) || (vals && !Ax)) return SPMVB200_ERR_INVALID;
    DISPATCH_OV(coo_to_csr_v, n_rows, nnz, rows, cols, vals, Ap, Aj, Ax, static_cast<cudaStream_t>(stream));
}

// ---- peer mapping --------------------------------------------------------------------------
int spmvb200_ipc_export(void *dev_ptr, unsigned char handle[SPMVB200_IPC_HANDLE_BYTES]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == SPMVB200_IPC_HANDLE_BYTES, "handle size");
    if (!dev_ptr || !handle) return SPMVB200_ERR_INVALID;
    cudaIpcMemHandle_t h;
    SPMV_CUDA_TRY(cudaIpcGetMemHandle(&h, dev_ptr));
    std::memcpy(handle, &h, sizeof(h));
    return SPMVB200_OK;
}
int spmvb200_ipc_open(const unsigned char handle[SPMVB200_IPC_HANDLE_BYTES], void **dev_ptr) {
    if (!handle || !dev_ptr) return SPMVB200_ERR_INVALID;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof(h));
    SPMV_CUDA_TRY(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return SPMVB200_OK;
}
int spmvb200_ipc_close(void *dev_ptr) {
    if (!dev_ptr) return SPMVB200_ERR_INVALID;
    SPMV_CUDA_TRY(cudaIpcCloseMemHandle(dev_ptr));
    return SPMVB200_OK;
}

}  // extern "C"
