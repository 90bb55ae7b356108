/*
 * spmv_b200.h -- C ABI of the B200 (sm_100a) CSR SpMV library, libspmvb200.so.
 *
 * This is the drop-in boundary for the reference's SpMV hot path.  Each typed entry
 * point below is what one instantiation of a reference kind
 *
 *     template <index_t, offset_t, mat_value_t, vec_x_value_t, vec_y_value_t>
 *     void SpMV_xxx(index_t n_rows, index_t n_cols, offset_t nnz,
 *                   const offset_t *Ap, const index_t *Aj, const mat_value_t *Ax,
 *                   const vec_x_value_t *x, vec_y_value_t *y);
 *
 * (reference/include/spmv/cusp/cusp.cuh:227-230, LightSpMV.cuh:379,
 *  merge_based/merge_based.cuh:22, cusparse.cuh:37-40; dispatched from
 *  reference/include/spmv.h:29-48) binds to.  include/spmv.h in this repository holds
 * the templates that forward to these symbols, so `SpMV(kind_str, ...)` keeps the
 * reference signature.
 *
 * Contract (SURVEY.md section 8(b)):
 *   - all five arrays are DEVICE pointers owned by the caller; Ap, Aj, Ax, x are
 *     read-only; y (n_rows entries) is fully overwritten: y = A*x (alpha = 1, beta = 0),
 *     empty rows give 0; n_rows == 0 is a no-op; n_cols == 0 (then nnz must be 0) writes
 *     y = 0 like any other matrix of empty rows -- the reference returns without touching y
 *     there (merge_based/dispatch_spmv_orig.cuh:564-570), which leaves y stale;
 *   - index type is int32; offsets are int32 (o32) or int64 (o64); values, x and y share
 *     one type, float (f32) or double (f64);
 *   - Ap, Aj, Ax must be 16-byte aligned (cudaMalloc gives 256); checked, not assumed:
 *     SPMVB200_ERR_ALIGNMENT otherwise;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = the legacy
 *     default stream) and the call returns without synchronising;
 *   - the return value is 0 or an SPMVB200_ERR_* code; nothing is printed, nothing
 *     aborts: include/spmv.h turns a non-zero status into the reference's
 *     print-and-exit behaviour (reference/include/common.cuh:13-23, spmv.h:46-47);
 *   - one host thread per (device, stream) at a time; scratch (tile coordinates, carries,
 *     row counter, row statistics) is cached inside the library per (device, stream);
 *   - there is NO CPU fallback: without a CUDA device every call returns
 *     SPMVB200_ERR_CUDA.
 */
#ifndef SPMV_B200_H_
#define SPMV_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPMVB200_API __attribute__((visibility("default")))

typedef void *spmvb200_stream_t; /* cudaStream_t */

enum {
    SPMVB200_OK = 0,
    SPMVB200_ERR_INVALID = 1,   /* negative size, NULL pointer with non-zero size */
    SPMVB200_ERR_ALIGNMENT = 2, /* Ap / Aj / Ax not 16-byte aligned */
    SPMVB200_ERR_CUDA = 3,      /* a CUDA runtime call failed; see spmvb200_last_cuda_error */
    SPMVB200_ERR_UNSUPPORTED = 4,
    SPMVB200_ERR_CUSPARSE = 5
};

/* kinds: the new SPMV_KINDS labels */
enum {
    SPMVB200_KIND_MERGE = 0,  /* "merge":  merge-path tiles + partition + carry fixup     */
    SPMVB200_KIND_VECTOR = 1, /* "vector": CSR-vector, sub-warp per row, shuffle reduce   */
    SPMVB200_KIND_LIGHT = 2,  /* "light":  LightSpMV-style dynamic row hand-out (atomics) */
    SPMVB200_KIND_AUTO = 3,   /* "auto":   host selector from cached row statistics       */
    SPMVB200_KIND_CUSPARSE = 4, /* "cusparse": cusparseSpMV baseline, setup hoisted        */
    SPMVB200_KIND_STREAM = 5  /* "stream": CSR-stream, TMA-staged row tiles, thread per row */
};

SPMVB200_API const char *spmvb200_status_string(int status);
SPMVB200_API const char *spmvb200_last_cuda_error(void);
SPMVB200_API const char *spmvb200_version(void);

/* ---- the hot path: one symbol per (kind, offset type, value type) ------------------ */
#define SPMVB200_DECLARE(KIND, OTAG, OFF_T, VTAG, VAL_T)                                   \
    SPMVB200_API int spmvb200_##KIND##_i32_##OTAG##_##VTAG(                                \
        int32_t n_rows, int32_t n_cols, OFF_T nnz, const OFF_T *Ap, const int32_t *Aj,    \
        const VAL_T *Ax, const VAL_T *x, VAL_T *y, spmvb200_stream_t stream);
#define SPMVB200_DECLARE_KIND(KIND)                       \
    SPMVB200_DECLARE(KIND, o32, int32_t, f32, float)      \
    SPMVB200_DECLARE(KIND, o32, int32_t, f64, double)     \
    SPMVB200_DECLARE(KIND, o64, int64_t, f32, float)      \
    SPMVB200_DECLARE(KIND, o64, int64_t, f64, double)

/* replaces SpMV_merge_based / SpMV_merge_based_generalized / SpMV_cub_merge_based
 * (reference/include/spmv/merge_based/merge_based.cuh:22, merge_genl/merge_genl.cuh:41,
 *  cub_merge.cuh:20) */
SPMVB200_DECLARE_KIND(merge)
/* replaces SpMV_cusp_origin / SpMV_cusp_warp_reduce / SpMV_cusp_warp_read_reduce
 * (reference/include/spmv/cusp/cusp.cuh:227, cusp_warp_reduce.cuh:138,
 *  cusp_warp_read_reduce.cuh:144) */
SPMVB200_DECLARE_KIND(vector)
/* replaces SpMV_light_vector / SpMV_light_warp (reference/include/spmv/LightSpMV.cuh:379,399) */
SPMVB200_DECLARE_KIND(light)
/* the short-regular-row case of SpMV_cusp_* (THREADS_PER_VECTOR = 2 / 4,
 * reference/include/spmv/cusp/cusp.cuh:189-203): persistent CTAs, row tiles staged in shared
 * memory with TMA bulk copies, one thread per row */
SPMVB200_DECLARE_KIND(stream)
/* new: per-matrix selector (BASELINE.json north_star "host-side selector") */
SPMVB200_DECLARE_KIND(auto)
/* replaces SpMV_cusparse (reference/include/spmv/cusparse.cuh:37-88); comparison baseline */
SPMVB200_DECLARE_KIND(cusparse)

/* Untyped form of the same call, for bindings that carry the types as data
 * (ctypes, the multi-GPU driver).  offset_bits in {32, 64}, value_bits in {32, 64}.
 * alpha_dev: optional DEVICE pointer to one value-typed scalar; y = (*alpha_dev) * A*x.
 * NULL means 1.  (merge_based/agent_spmv_orig.cuh:425-433 carries alpha the same way.)
 * y_peers / n_peers: optional array (HOST memory) of extra DEVICE pointers that receive the
 * same y stores (peer-mapped buffers of other GPUs; the fused SpMV + all-gather of the
 * row-sharded power iteration).  Each is indexed like y.  Supported by merge/vector/light.
 * Only rows that have nonzeros are stored to the peers (an empty row's y is always 0), so the
 * peer buffers must hold 0 at the positions of empty rows -- zero them once.
 * n_peers == -1: y_peers[0] is an NVLink multicast address (NVLS; e.g. the multicast_ptr of a
 * torch symmetric-memory buffer) and every such row is stored once with multimem.st. */
/* Generalised SpMV  y[r] = REDUCE_k COMBINE(Ax[k], x[Aj[k]])  from IDENTITY: the fixed menu that
 * stands in for the template functor of the reference's SpMV_merge_based_generalized
 * (merge_genl/merge_genl.cuh:19-38, cpu_navie.hpp:20-35).  Served by the merge-path kernel only
 * (kind merge or auto), as in the reference.  Empty rows yield IDENTITY.
 * Min-plus and max-plus with infinite x (an unreached vertex is x = +inf) follow IEEE; when a
 * combine yields NaN (+inf + -inf, or a NaN input) the result is unspecified: it depends on where
 * the NaN meets the reduction (min(u, v) as u < v ? u : v forgets a NaN once a later term comes). */
enum {
    SPMVB200_SEMIRING_PLUS_TIMES = 0, /* 0,    a*x,            u+v        (ordinary SpMV)     */
    SPMVB200_SEMIRING_MIN_PLUS = 1,   /* +inf, a+x,            min(u,v)   (shortest paths)    */
    SPMVB200_SEMIRING_MAX_PLUS = 2,   /* -inf, a+x,            max(u,v)   (longest paths)     */
    SPMVB200_SEMIRING_OR_AND = 3      /* 0,    a!=0 && x!=0,   max(u,v)   (reachability, 0/1) */
};
/* beta_dev: optional DEVICE pointer to one value-typed scalar: y = alpha*A*x + beta*y (plus-times
 * only; merge-path kernel; merge_based/agent_spmv_orig.cuh:425-433 HAS_BETA).  NULL means 0 and y
 * is not read.  Fields after `stream` default to plus-times / no beta when zero-initialised.
 * flags: SPMVB200_FLAG_STATIC_PATTERN -- the caller vouches that Ap (same pointer, n_rows, nnz)
 * still holds what it held at the previous call on this stream, so the merge-path kernel may
 * reuse that call's tile coordinates instead of searching again (an iterative solver's matrix;
 * the reference re-derives everything per call, merge_based/dispatch_spmv_orig.cuh:613-660).
 * The first call on a matrix, or any call after Ap's contents changed, must not pass it.
 * Special values (every kind, SpMM and the beta form): Inf and NaN propagate per IEEE within their
 * own row only -- a row is NaN if one of its products is NaN or it has both a +inf and a -inf
 * product, else +-inf if it has a product of that sign -- and never reach another row.  Stored
 * zeros are multiplied, as cuSPARSE does: 0 * inf in a row makes it NaN.  Subnormal values are
 * kept (the library is not built to flush them to zero). */
#define SPMVB200_FLAG_STATIC_PATTERN 1
typedef struct {
    int32_t kind;
    int32_t offset_bits;
    int32_t value_bits;
    int32_t n_peers;
    int64_t n_rows;
    int64_t n_cols;
    int64_t nnz;
    const void *Ap;
    const int32_t *Aj;
    const void *Ax;
    const void *x;
    void *y;
    const void *alpha_dev;
    void *const *y_peers;
    spmvb200_stream_t stream;
    int32_t semiring;
    int32_t flags;
    const void *beta_dev;
} spmvb200_args_t;
SPMVB200_API int spmvb200_spmv(const spmvb200_args_t *args);

/* ---- K right-hand sides at once (SpMM), K in {2, 4, 8} -----------------------------------
 * Y = alpha * A * X with X [n_cols x k] and Y [n_rows x k] row-major with leading dimensions
 * ldx, ldy (in elements).  New with respect to the reference (SURVEY.md 8(f) rank 4); the only
 * way past the gather bound of CSR SpMV: one gather returns k values.  X and Y must be 16-byte
 * aligned (8 for k = 2 floats) and ldx, ldy must keep every row so aligned, else
 * SPMVB200_ERR_ALIGNMENT.  alpha_dev as in spmvb200_spmv. */
typedef struct {
    int32_t offset_bits;
    int32_t value_bits;
    int32_t k;
    int32_t reserved;
    int64_t n_rows;
    int64_t n_cols;
    int64_t nnz;
    const void *Ap;
    const int32_t *Aj;
    const void *Ax;
    const void *X;
    int64_t ldx;
    void *Y;
    int64_t ldy;
    const void *alpha_dev;
    spmvb200_stream_t stream;
} spmvb200_spmm_args_t;
SPMVB200_API int spmvb200_spmm(const spmvb200_spmm_args_t *args);

/* ---- conjugate-gradient solve A x = b on the device (csrc/cg.cu) ---------------------------
 * A is n x n, symmetric positive definite, in CSR; preconditioned CG (Hestenes-Stiefel) with
 * M = I, or M = diag(A) with SPMVB200_CG_JACOBI.  One iteration is one SpMV of `kind` (any kind
 * spmvb200_spmv accepts; SPMVB200_FLAG_STATIC_PATTERN on every call after the first) and three
 * streaming kernels.  Dot products accumulate in double in a fixed order, so a solve is
 * deterministic for the deterministic kinds.  Stops after the first iteration with
 * ||r|| <= rtol * ||b|| (r the recursive residual), after max_iter iterations, or at a breakdown
 * (p.q <= 0 or not finite: A is not SPD); a breakdown is not an error.  x holds the initial guess
 * on entry and the solution on return; b = 0 gives x = 0.  residual_norm is ||b - A x|| of the
 * returned x, computed once more in fp64.  The host reads the device flags once per batch of
 * iterations (1, 2, 4, ... 64), not per iteration.  Enqueued on `stream`; synchronises before it
 * returns.  Workspace (3 vectors, 5 with Jacobi) is cached per (device, stream) like the other
 * scratch and freed by spmvb200_release_cache.  Errors: SPMVB200_ERR_INVALID for an unknown kind
 * or flag, rtol <= 0 or NaN, max_iter < 0, a NULL pointer with n > 0, x == b, or (Jacobi) a row
 * whose diagonal entry is missing or zero; the alignment rules of spmvb200_spmv. */
#define SPMVB200_CG_JACOBI 1
typedef struct {
    int32_t kind, offset_bits, value_bits, flags; /* flags: 0 or SPMVB200_CG_JACOBI */
    int64_t n, nnz;                               /* A is n x n */
    const void *Ap;
    const int32_t *Aj;
    const void *Ax;
    const void *b;
    void *x; /* initial guess in, solution out (DEVICE) */
    double rtol;
    int64_t max_iter;
    spmvb200_stream_t stream;
} spmvb200_cg_args_t;
typedef struct {
    int64_t iterations;
    double residual_norm;
    double b_norm;
    int32_t converged;
    int32_t breakdown;
} spmvb200_cg_result_t;
SPMVB200_API int spmvb200_cg(const spmvb200_cg_args_t *args, spmvb200_cg_result_t *out);

/* ---- BiCGSTAB solve A x = b on the device (csrc/bicgstab.cu) -------------------------------
 * A is n x n in CSR and need not be symmetric; right-preconditioned BiCGSTAB (van der Vorst) with
 * M = I, or M = diag(A) with SPMVB200_CG_JACOBI, in the operation order of
 * scipy.sparse.linalg.bicgstab.  Takes the records of spmvb200_cg (spmvb200_cg_args_t,
 * spmvb200_cg_result_t) with the same meaning, the same argument checks and status codes; n == 0
 * reports convergence after 0 iterations.  One iteration is two SpMVs of `kind`
 * (SPMVB200_FLAG_STATIC_PATTERN on every call after the first) and five streaming kernels; dot
 * products accumulate in double in a fixed order, so a solve is deterministic for the
 * deterministic kinds.  `iterations` counts the times x was moved along the search direction, so
 * a solve that converges at the half step (||s|| <= rtol * ||b||) counts that iteration.  It stops
 * when the recursive residual meets ||r|| <= rtol * ||b|| (or ||s|| does), after max_iter
 * iterations, or at a breakdown: an exact zero or a non-finite value of (r^, r), (r^, v), alpha,
 * (t, t) or omega, or omega == 0 -- the method cannot continue (e.g. (r^, v) = 0 for the shadow
 * residual r^ = r0), or the input holds NaN or inf.  A breakdown is not an error; x is then the
 * last finite iterate.  residual_norm is ||b - A x|| of the returned x, computed once more in
 * fp64.  Workspace (5 vectors, 8 with Jacobi) is cached per (device, stream) and freed by
 * spmvb200_release_cache. */
SPMVB200_API int spmvb200_bicgstab(const spmvb200_cg_args_t *args, spmvb200_cg_result_t *out);

/* ---- restarted GMRES(m) solve A x = b on the device (csrc/gmres.cu) ------------------------
 * A is n x n in CSR and need not be symmetric; right-preconditioned GMRES(m) with M = I, or
 * M = diag(A) with SPMVB200_CG_JACOBI: it solves A M^-1 u = b, x = x0 + M^-1 V y, so the residual
 * it minimises over each Krylov space is the true residual b - A x and rtol means what it means
 * for spmvb200_cg.  (scipy.sparse.linalg.gmres preconditions on the left.)  Takes the records of
 * spmvb200_cg with the same meaning, the same argument checks and status codes, and
 * SPMVB200_ERR_INVALID for `restart` outside [1, SPMVB200_GMRES_MAX_RESTART], checked before any
 * CUDA call; the cycle length used is m = min(restart, n).  n == 0 reports convergence after 0
 * iterations.  An Arnoldi step is one SpMV of `kind` (SPMVB200_FLAG_STATIC_PATTERN on every call
 * after the first) and four streaming kernels, whatever the step's place in the cycle: classical
 * Gram-Schmidt with one re-orthogonalisation (CGS2), dot products in double in a fixed order, the
 * Hessenberg matrix and its Givens rotations (r = hypot(a, b)) in double on the device.  A cycle
 * ends after m steps, when the residual estimate |g_{j+1}| <= rtol * ||b||, at a lucky breakdown
 * (||w|| after the orthogonalisation <= eps * ||w|| before it, eps of the value type), or at
 * max_iter; then x += M^-1 V y, and the explicit ||b - A x|| decides convergence, or the next
 * cycle starts from that residual.  A breakdown (not an error) is a non-finite h, norm or
 * rotation (x is left at the start of that cycle), a non-finite ||b|| or ||r0|| (NaN or inf in
 * the input), or a lucky breakdown whose explicit residual still misses the tolerance.
 * `iterations` counts Arnoldi steps (the SpMVs inside cycles).  The host reads the device flags
 * once per batch of 1, 2, 4, ... 64 steps; a cycle that ends early on the device leaves the rest
 * of its m steps idle, and those count against max_iter.  residual_norm is ||b - A x|| of the
 * returned x, computed once more in fp64.  Workspace ((m + 1) vectors, m + 3 with Jacobi) is
 * cached per (device, stream) and freed by spmvb200_release_cache. */
#define SPMVB200_GMRES_MAX_RESTART 64
SPMVB200_API int spmvb200_gmres(const spmvb200_cg_args_t *args, int32_t restart, spmvb200_cg_result_t *out);

/* ---- merge-path partition, exposed so parity tests can demand bit-exact coordinates --- */
/* Row coordinate of the merge path on each diagonal min(t * tile_items, n_rows + nnz),
 * t = 0 .. n_coords-1, written to the DEVICE array coords_x (int32).  The nonzero
 * coordinate is diagonal - coords_x[t].
 * Replaces DeviceSpmvSearchKernel (reference/include/spmv/merge_based/dispatch_spmv_orig.cuh:109-148)
 * and SearchMergePath (merge_based/thread_search.cuh:16-49). */
SPMVB200_API int spmvb200_merge_path_partition_o32(int32_t n_rows, int32_t nnz, const int32_t *Ap,
                                                   int64_t tile_items, int64_t n_coords,
                                                   int32_t *coords_x, spmvb200_stream_t stream);
SPMVB200_API int spmvb200_merge_path_partition_o64(int32_t n_rows, int64_t nnz, const int64_t *Ap,
                                                   int64_t tile_items, int64_t n_coords,
                                                   int32_t *coords_x, spmvb200_stream_t stream);
/* tile size (merge items per thread block) the merge kernel uses for this type pair */
SPMVB200_API int64_t spmvb200_merge_tile_items(int offset_bits, int value_bits);

/* nnz-balanced row split for `parts` shards (SURVEY.md 8(e)): row_bounds (HOST, parts+1
 * int64) from the merge path on diagonals floor(g*(n_rows+nnz)/parts).  Synchronises. */
SPMVB200_API int spmvb200_row_split_o32(int32_t n_rows, int32_t nnz, const int32_t *Ap, int parts,
                                        int64_t *row_bounds, spmvb200_stream_t stream);
SPMVB200_API int spmvb200_row_split_o64(int32_t n_rows, int64_t nnz, const int64_t *Ap, int parts,
                                        int64_t *row_bounds, spmvb200_stream_t stream);

/* Weighted form of the same search, for splits that weigh a row differently from a nonzero or
 * that are re-balanced from measured shard times (spmv_samples_b200/dist.py): with
 * f(r) = w_den*Ap[r] + w_num*r the cost of the first r rows (w_num/w_den = cost of a row in
 * nonzeros; 1/1 is the merge path above), rows_out[k] = max{ r in [0, n_rows] : f(r) <= targets[k] }.
 * targets / rows_out are HOST arrays of n_targets int64; 0 <= w_num, 1 <= w_den, both <= 2^20.
 * Synchronises. */
SPMVB200_API int spmvb200_rows_at_cost_o32(int32_t n_rows, const int32_t *Ap, int64_t w_num,
                                           int64_t w_den, int n_targets, const int64_t *targets,
                                           int64_t *rows_out, spmvb200_stream_t stream);
SPMVB200_API int spmvb200_rows_at_cost_o64(int32_t n_rows, const int64_t *Ap, int64_t w_num,
                                           int64_t w_den, int n_targets, const int64_t *targets,
                                           int64_t *rows_out, spmvb200_stream_t stream);

/* ---- row statistics + selector --------------------------------------------------------- */
typedef struct {
    int64_t n_rows;
    int64_t nnz;
    int64_t max_row_len;
    int64_t empty_rows;
    double mean_row_len;
    double std_row_len;
    int32_t chosen_kind;  /* what "auto" runs for this matrix */
    int32_t chosen_width; /* lanes per row for vector / light */
} spmvb200_row_stats_t;
/* One pass over Ap on the device; synchronises the stream.  This call always recomputes (and
 * refreshes the cache); the "auto" kind reuses the cached result keyed on (Ap, n_rows, nnz). */
SPMVB200_API int spmvb200_row_stats(int offset_bits, int64_t n_rows, int64_t nnz, const void *Ap,
                                    spmvb200_row_stats_t *out, spmvb200_stream_t stream);

/* ---- tunables (benchmarking / ablation); names in DESIGN.md --------------------------- */
SPMVB200_API int spmvb200_set_option(const char *name, int64_t value);
SPMVB200_API int64_t spmvb200_get_option(const char *name);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
SPMVB200_API int64_t spmvb200_launch_count(void);
/* drop cached scratch / statistics (all devices) */
SPMVB200_API void spmvb200_release_cache(void);

/* Measurement aid (csrc/diag.cu): `gathers` uniformly random 4-byte gathers of an x of
 * `x_elements` floats, the index stream read as the kernels read Aj -- the gather rate every CSR
 * kernel that gathers x through L1 is bounded by.  Best of `reps` launches, in milliseconds. */
SPMVB200_API int spmvb200_gather_yardstick(int64_t x_elements, int64_t gathers, int reps,
                                           spmvb200_stream_t stream, double *best_ms);

/* The hot-x plan of the merge-path kernel (csrc/hotx.cu): for an x far longer than the TLB and L2
 * reach (option "hot_x_min_bytes", 256 MB) and a caller that passes SPMVB200_FLAG_STATIC_PATTERN,
 * the library keeps a copy of Aj in which the most frequent columns are renumbered into one dense
 * array x_hot (refilled from x before every SpMV).  Products and their order are unchanged: y is
 * bit-identical.  Costs nnz * 4 bytes of device memory, built at the first flagged call.  Reports
 * what was built for this Aj on the current device (0 columns = no plan).  The flag therefore
 * vouches for Aj as well as Ap.  If the device has no room for the plan, the calls proceed without it.  Callers behind the reference's SpMV(kind_str, ...) signature,
 * which has no flags, vouch through option "assume_static_pattern" = 1 (main.cu does for its
 * timing loop).  Nothing in the reference corresponds (it gathers x[Aj[k]] as is,
 * merge_based/agent_spmv_orig.cuh:474-506). */
SPMVB200_API int spmvb200_hot_x_info(const int32_t *Aj, int64_t *hot_columns, double *hot_share,
                                     double *build_ms);
/* The first `table_columns` ranks of that plan are its most frequent columns: the persistent form
 * of the merge-path tile kernel (one CTA per SM walking over tiles) keeps their x values in a
 * shared-memory table, where a gather costs a ninth of an L1 gather (options "hot_x_table",
 * "hot_x_table_bytes").  With it the plan is also built for a short x (then all hot columns are
 * table columns).  table_share: the fraction of the gathers they receive. */
SPMVB200_API int spmvb200_hot_x_table_info(const int32_t *Aj, int64_t *table_columns, double *table_share);

/* ---- host-buffer convenience: the end-to-end call --------------------------------------
 * A CSR matrix uploaded once (as reference/main.cu:55-69 does), then y = A*x with x and y
 * in HOST memory: H2D copy of x, kernel, D2H copy of y, stream synchronised on return. */
typedef struct spmvb200_matrix spmvb200_matrix_t;
SPMVB200_API int spmvb200_matrix_create(int offset_bits, int value_bits, int64_t n_rows,
                                        int64_t n_cols, int64_t nnz, const void *Ap_host,
                                        const int32_t *Aj_host, const void *Ax_host,
                                        spmvb200_matrix_t **out);
/* Same object over CSR arrays that already live on the device (borrowed, never freed). */
SPMVB200_API int spmvb200_matrix_create_from_device(int offset_bits, int value_bits, int64_t n_rows,
                                                    int64_t n_cols, int64_t nnz, const void *Ap_dev,
                                                    const int32_t *Aj_dev, const void *Ax_dev,
                                                    spmvb200_matrix_t **out);
SPMVB200_API int spmvb200_matrix_spmv_host(spmvb200_matrix_t *m, int kind, const void *x_host,
                                           void *y_host);
/* Pipelined form for a sequence of independent right-hand sides: SPMVB200_MAX_SLOTS slots
 * (0 .. MAX-1), each with its own stream and device x/y (created on first use).  submit enqueues
 * H2D(x) -> SpMV -> D2H(y) on the slot's stream and returns; wait blocks until that slot's y_host
 * is complete.  Cycling through the slots overlaps one call's upload with another's kernel and a
 * third's download (both copy engines + the SMs busy): a step is upload + kernel + download long,
 * so three slots are what it takes to hide both copies behind the kernel when each copy is
 * shorter than the kernel.  x_host / y_host should be pinned, and must stay untouched until the
 * slot has been waited on. */
#define SPMVB200_MAX_SLOTS 4
SPMVB200_API int spmvb200_matrix_submit_host(spmvb200_matrix_t *m, int kind, int slot,
                                             const void *x_host, void *y_host);
SPMVB200_API int spmvb200_matrix_wait(spmvb200_matrix_t *m, int slot);
SPMVB200_API void spmvb200_matrix_destroy(spmvb200_matrix_t *m);

/* ---- device-side data layer: synthetic generators and COO -> CSR ------------------------
 * Counter-based (splitmix64) so the host restatement in oracle/generators.py matches bit
 * for bit.  All pointers are DEVICE pointers. */
SPMVB200_API int spmvb200_gen_uniform_pm1(int value_bits, uint64_t seed, uint32_t stream_id,
                                          uint64_t first, int64_t count, void *out,
                                          spmvb200_stream_t stream);
SPMVB200_API int spmvb200_gen_lap2d(int offset_bits, int value_bits, int32_t grid_n, void *Ap,
                                    int32_t *Aj, void *Ax, spmvb200_stream_t stream);
SPMVB200_API int spmvb200_gen_uniform_rows(int offset_bits, int value_bits, int32_t n_rows,
                                           int32_t n_cols, int32_t row_len, uint64_t seed,
                                           void *Ap, int32_t *Aj, void *Ax,
                                           spmvb200_stream_t stream);
SPMVB200_API int spmvb200_gen_rmat_edges(int32_t scale, uint64_t seed, uint64_t first_edge,
                                         int64_t count, int32_t *rows, int32_t *cols,
                                         spmvb200_stream_t stream);
/* Stable COO -> CSR (input order kept within a row, duplicates kept), 64-bit safe.
 * Replaces ToCsr (reference/include/load.hpp:420-474).  rows/cols are clobbered (used as
 * sort buffers); vals may be NULL (pattern only: Aj and Ap written).  Allocates its own
 * temporaries and synchronises. */
SPMVB200_API int spmvb200_coo_to_csr(int offset_bits, int value_bits, int32_t n_rows, int64_t nnz,
                                     int32_t *rows, int32_t *cols, const void *vals, void *Ap,
                                     int32_t *Aj, void *Ax, spmvb200_stream_t stream);

/* ---- power iteration helpers (the row-sharded iterated SpMV of BASELINE.json configs[4]) --
 * sumsq_dev (DEVICE, one double) = sum of v[i]^2, deterministic two-pass reduction;
 * alpha_dev (DEVICE, one value-typed scalar) = 1 / sqrt(*sumsq_dev), or 1 if the sum is 0. */
SPMVB200_API int spmvb200_sum_squares(int value_bits, int64_t n, const void *v, double *sumsq_dev,
                                      spmvb200_stream_t stream);
SPMVB200_API int spmvb200_inv_sqrt(int value_bits, const double *sumsq_dev, void *alpha_dev,
                                   spmvb200_stream_t stream);

/* Everything between two SpMVs of the row-sharded power iteration in ONE kernel: sum of squares
 * of this rank's `n` values of y, exchange of the per-rank sums, *sumsq_dev = their total (added
 * in rank order: the same bits on every rank), *alpha_dev = 1 / sqrt(total).  Mailboxes:
 * SPMVB200_MAILBOX_BYTES of device memory per rank, filled with the double -1.0 once before the
 * first step, each mapped into every other rank (cudaIpc / peer access / symmetric memory).
 * mailbox_of_rank[q] (HOST array of `world` DEVICE pointers) is rank q's mailbox as addressed
 * from this rank, [rank] being mailbox_local itself; or mailbox_multicast is one NVLink multicast
 * address that reaches all of them (then mailbox_of_rank may be NULL).  `step` counts up from 0
 * by one per call, in step on all ranks.  Leaving the kernel means every rank has finished the
 * kernels it enqueued before its own call for this step -- the step barrier of the fused
 * exchange.  A rank that does not arrive within ~4 s sets *error_dev (DEVICE int, zero it once)
 * to 1 + its number on the ranks that waited for it, instead of hanging them.
 * The reference has no iteration and no exchange (main.cu:102-113 repeats one call). */
#define SPMVB200_MAILBOX_BYTES 256
SPMVB200_API int spmvb200_norm_exchange(int value_bits, int64_t n, const void *y_local, int rank,
                                        int world, uint64_t step, void *mailbox_local,
                                        void *const *mailbox_of_rank, void *mailbox_multicast,
                                        double *sumsq_dev, void *alpha_dev, int *error_dev,
                                        spmvb200_stream_t stream);

/* ---- the row-sharded power iteration from ONE process (csrc/multi.cu) ----------------------
 * BASELINE.json's multi-GPU configuration for a C / C++ host (main.cu --gpus N): no Python, no
 * torch.distributed, no NCCL.  The matrix (square) is cut into `n_gpus` row blocks at the merge
 * path's nnz-balanced boundaries; GPU g keeps its block and two full-length replicas of x; a step
 * is the SpMV of the local rows, whose row stores also go into every other GPU's replica of the
 * next x through peer access over NVLink (the all-gather is the kernel's epilogue), followed by
 * spmvb200_norm_exchange (norm, alpha and step barrier in one kernel).  devices = NULL means
 * 0 .. n_gpus-1; every pair must be peer-accessible (SPMVB200_ERR_UNSUPPORTED otherwise).
 * create_from_device takes CSR arrays resident on devices[0] (not kept: each GPU gets its own
 * copy of its rows); create takes HOST arrays.  steps enqueues and returns; run times `steps`
 * steps on the devices (the slowest GPU counts) and synchronises; get returns the current
 * iterate (n values, HOST, may be NULL), ||A x_k|| of the last step and the n_gpus + 1 row
 * boundaries (HOST int64, may be NULL). */
typedef struct spmvb200_power spmvb200_power_t;
SPMVB200_API int spmvb200_power_create(int n_gpus, const int *devices, int offset_bits, int value_bits,
                                       int64_t n_rows, int64_t nnz, const void *Ap_host,
                                       const int32_t *Aj_host, const void *Ax_host, int kind,
                                       spmvb200_power_t **out);
SPMVB200_API int spmvb200_power_create_from_device(int n_gpus, const int *devices, int offset_bits,
                                                   int value_bits, int64_t n_rows, int64_t nnz,
                                                   const void *Ap_dev, const int32_t *Aj_dev,
                                                   const void *Ax_dev, int kind, spmvb200_power_t **out);
SPMVB200_API int spmvb200_power_reset(spmvb200_power_t *p);
SPMVB200_API int spmvb200_power_steps(spmvb200_power_t *p, int steps);
SPMVB200_API int spmvb200_power_run(spmvb200_power_t *p, int steps, double *ms_per_step);
SPMVB200_API int spmvb200_power_sync(spmvb200_power_t *p);
SPMVB200_API int spmvb200_power_get(spmvb200_power_t *p, void *x_host, double *norm, int64_t *row_bounds);
/* 0: the replicas of x are fed by peer stores (or there is one GPU); 1: by one multimem.st per row
 * through an NVLink multicast object (csrc/mcast.cu).  Option "power_exchange": 0 / 1 force one
 * (1 fails with SPMVB200_ERR_UNSUPPORTED where there is no multicast), -1 = multicast where the
 * box has it, peer stores otherwise. */
SPMVB200_API int spmvb200_power_exchange(const spmvb200_power_t *p);
SPMVB200_API void spmvb200_power_destroy(spmvb200_power_t *p);

/* ---- device timing of the dominant kernel (bench.py's roofline.achieved) ------------------
 * With option "time_main_kernel" = 1 every merge / vector / light call brackets its main
 * kernel with cudaEvents on the caller's stream.  This call synchronises on them, returns the
 * summed milliseconds and the number of launches since the last call, and resets both. */
SPMVB200_API int spmvb200_main_kernel_time(double *total_ms, int64_t *launches);

/* ---- plain device memory (cudaMalloc), exportable with spmvb200_ipc_export ---------------- */
SPMVB200_API int spmvb200_device_malloc(size_t bytes, void **dev_ptr);
SPMVB200_API int spmvb200_device_free(void *dev_ptr);

/* ---- peer mapping for the fused SpMV + all-gather (one process per GPU) ---------------- */
#define SPMVB200_IPC_HANDLE_BYTES 64
SPMVB200_API int spmvb200_ipc_export(void *dev_ptr, unsigned char handle[SPMVB200_IPC_HANDLE_BYTES]);
SPMVB200_API int spmvb200_ipc_open(const unsigned char handle[SPMVB200_IPC_HANDLE_BYTES],
                                   void **dev_ptr);
SPMVB200_API int spmvb200_ipc_close(void *dev_ptr);

#ifdef __cplusplus
}
#endif
#endif /* SPMV_B200_H_ */
