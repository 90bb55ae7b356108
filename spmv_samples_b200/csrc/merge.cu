// merge.cu -- merge-path CSR SpMV for sm_100a: partition kernel, tile kernel, carry fixup.
//
// What it computes is what the reference's vendored CUB 1.15 merge-based SpMV computes
// (reference/include/spmv/merge_based/dispatch_spmv_orig.cuh:109-229,
//  agent_spmv_orig.cuh:454-760, agent_segment_fixup.cuh:229-358, thread_search.cuh:16-49):
// the (row-end, nonzero) merge path of length n_rows + nnz is cut into equal tiles by a
// binary-search partition kernel, each tile reduces its nonzeros into the rows that end inside
// it and hands the unfinished tail to a fixup pass.  How a tile is processed is new, because
// a B200 SM has ~4x the HBM bandwidth per SM of the parts CUB's agent was tuned for and the
// agent's per-thread path search + serial merge (about 45 scalar shared-memory operations per
// thread) is shared-memory-issue bound here (first ncu capture: mio_throttle + short
// scoreboard dominant, 75 thread instructions per path item, 16 % of the HBM roofline):
//   * a tile is 1020 path items (128 threads; the TMA-staged ablation kernel keeps 256 / 2044);
//   * every thread owns 8 consecutive nonzeros: 128-bit evict-first loads of Aj and Ax from a
//     16-byte aligned position straight into registers, x gathered with an L2 evict-last
//     policy, products kept in registers (merge_tile_reg_body, the default).  The first version
//     staged the tile's Ap / Aj / Ax segments in shared memory with TMA 1-D bulk copies
//     (merge_tile_tma_kernel, option merge_staging = 1, kept under test as the ablation): the
//     27-35 KB per CTA it takes come out of the L1 that holds the x gathers in flight, and it
//     is 1.1x (int32 offsets) to 2.9x (R-MAT scale 27) slower -- DESIGN.md section 3, point 2;
//   * rows are delimited by a byte flag per nonzero, scattered one thread per row end; the
//     reduction is a segmented scan (serial in the thread, shuffles across the warp, one
//     shared-memory hop across warps) -- no per-thread merge-path search at all;
//   * the scanned values go to shared memory once, and one thread per row end picks its
//     row's total, so y is written coalesced;
//   * only the row coordinate of each tile boundary is stored (int32); the nonzero
//     coordinate is diagonal - row, which keeps the scratch 64-bit safe for free;
//   * the tile carry-out goes to a fixup kernel that is deterministic (run-head threads sum
//     their run in tile order; no atomics, unlike agent_segment_fixup.cuh:257,269).
// Within a tile the work is bounded by construction (rows + nonzeros <= tile size), which is
// the load-balance guarantee of the merge path; the in-tile phases are regular on top of it.
#include <climits>

#include "common.cuh"

namespace spmvb200 {

namespace {

#ifndef SPMV_MERGE_BLOCK
#define SPMV_MERGE_BLOCK 256
#endif
constexpr int kMergeBlock = SPMV_MERGE_BLOCK;
constexpr int kMergeIPT = 8;
constexpr int kSlots = kMergeBlock * kMergeIPT;  // staged elements per array
constexpr int kMergeTile = kSlots - 4;           // path items per tile: room for the <=3-element
                                                 // align-down shift of the bulk copies
constexpr int kPad = 8;

template <typename OffT, typename ValT>
constexpr size_t merge_smem_bytes() {
    return 16 + (size_t)(kSlots + kPad) * sizeof(OffT) + (size_t)kSlots * (sizeof(int32_t) + sizeof(ValT) + 1);
}

// ---------------------------------------------------------------- partition (search) kernel
// thread t: row coordinate of the merge path on diagonal min(t*tile_items, n_rows+nnz).
template <typename OffT>
__global__ void __launch_bounds__(256)
merge_partition_kernel(int32_t n_rows, OffT nnz, const OffT *__restrict__ Ap, int64_t tile_items,
                       int64_t n_coords, int32_t *__restrict__ coords_x) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_coords) return;
    const int64_t total = (int64_t)n_rows + (int64_t)nnz;
    int64_t diag = t * tile_items;
    if (diag > total) diag = total;
    const OffT *__restrict__ row_end = Ap + 1;
    int64_t lo = diag - (int64_t)nnz > 0 ? diag - (int64_t)nnz : 0;
    int64_t hi = diag < n_rows ? diag : n_rows;
    while (lo < hi) {
        const int64_t pivot = (lo + hi) >> 1;
        if ((int64_t)__ldg(row_end + pivot) <= diag - pivot - 1) lo = pivot + 1;
        else hi = pivot;
    }
    coords_x[t] = (int32_t)lo;
}

// stage `count` elements of g[gbeg ...) into s[(gbeg - a0) ...), a0 = gbeg aligned down to V
// elements (V * sizeof(T) a multiple of 16): the aligned interior by one bulk copy (thread 0),
// the ragged tail (fewer than V elements, or a whole tiny segment) by plain loads.
struct StagePlan {
    int64_t a0;           // first element of the bulk copy (aligned)
    uint32_t bulk_elems;  // 0 = no bulk copy
    int64_t tail_beg;     // first element loaded by threads
    int tail_cnt;
    int shift;            // gbeg - a0
};
template <int V>
__device__ __forceinline__ StagePlan plan_stage(int64_t gbeg, int count) {
    StagePlan p;
    p.a0 = gbeg & ~(int64_t)(V - 1);
    p.shift = (int)(gbeg - p.a0);
    const int64_t gend = gbeg + count;
    const int64_t be = gend & ~(int64_t)(V - 1);
    if (be > p.a0 && count > 0) {
        p.bulk_elems = (uint32_t)(be - p.a0);
        p.tail_beg = be;
    } else {
        p.bulk_elems = 0;
        p.tail_beg = gbeg;
    }
    p.tail_cnt = (int)(gend - p.tail_beg);
    return p;
}

// 8 consecutive staged values -> registers (128-bit shared loads)
__device__ __forceinline__ void lds8(const float *s, float (&v)[8]) {
    const float4 a = *reinterpret_cast<const float4 *>(s);
    const float4 b = *reinterpret_cast<const float4 *>(s + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
    v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void lds8(const double *s, double (&v)[8]) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const double2 a = *reinterpret_cast<const double2 *>(s + 2 * k);
        v[2 * k] = a.x;
        v[2 * k + 1] = a.y;
    }
}
__device__ __forceinline__ void sts8(float *s, const float (&v)[8]) {
    *reinterpret_cast<float4 *>(s) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4 *>(s + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void sts8(double *s, const double (&v)[8]) {
#pragma unroll
    for (int k = 0; k < 4; ++k) *reinterpret_cast<double2 *>(s + 2 * k) = make_double2(v[2 * k], v[2 * k + 1]);
}

// ---------------------------------------------------------------------------- tile kernel
template <typename OffT, typename ValT>
__global__ void __launch_bounds__(kMergeBlock)
merge_tile_tma_kernel(int32_t n_rows, OffT nnz, const OffT *__restrict__ Ap,
                  const int32_t *__restrict__ Aj, const ValT *__restrict__ Ax,
                  const ValT *__restrict__ x, ValT *__restrict__ y,
                  const ValT *__restrict__ alpha_dev, PeerOut peers,
                  const int32_t *__restrict__ coords_x, int32_t *__restrict__ carry_row,
                  ValT *__restrict__ carry_val) {
    constexpr int IPT = kMergeIPT;
    constexpr int VR = 16 / sizeof(OffT);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw);
    OffT *s_rend = reinterpret_cast<OffT *>(smem_raw + 16);
    ValT *s_val = reinterpret_cast<ValT *>(s_rend + kSlots + kPad);
    int32_t *s_col = reinterpret_cast<int32_t *>(s_val + kSlots);
    unsigned char *s_flag = reinterpret_cast<unsigned char *>(s_col + kSlots);
    __shared__ ValT s_wval[kMergeBlock / 32];
    __shared__ int s_wflag[kMergeBlock / 32];

    const int tid = threadIdx.x;
    const int64_t tile = blockIdx.x;
    const int64_t total = (int64_t)n_rows + (int64_t)nnz;
    const int64_t d0 = tile * kMergeTile;
    const int64_t d1 = d0 + kMergeTile < total ? d0 + kMergeTile : total;
    const int32_t sx = __ldg(coords_x + tile);
    const int32_t ex = __ldg(coords_x + tile + 1);
    const int64_t sy = d0 - sx;
    const int R = ex - sx;                // rows that end inside this tile
    const int Z = (int)((d1 - ex) - sy);  // nonzeros inside this tile

    // Aj and Ax are staged with the same shift (sy mod 4), so slot s of either array holds
    // tile-local nonzero s - shift
    const StagePlan pr = plan_stage<VR>((int64_t)sx + 1, R);
    const StagePlan pc = plan_stage<4>(sy, Z);
    const int shift = pc.shift;

    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    // clear this thread's 8 row-start flags
    *reinterpret_cast<uint2 *>(s_flag + tid * IPT) = make_uint2(0u, 0u);
    __syncthreads();
    if (tid == 0) {
        const uint64_t pol = policy_evict_first();
        mbar_arrive_expect_tx(bar, pr.bulk_elems * (uint32_t)sizeof(OffT) +
                                       pc.bulk_elems * (uint32_t)(sizeof(int32_t) + sizeof(ValT)));
        if (pr.bulk_elems) bulk_g2s(s_rend, Ap + pr.a0, pr.bulk_elems * (uint32_t)sizeof(OffT), bar, pol);
        if (pc.bulk_elems) {
            bulk_g2s(s_col, Aj + pc.a0, pc.bulk_elems * (uint32_t)sizeof(int32_t), bar, pol);
            bulk_g2s(s_val, Ax + pc.a0, pc.bulk_elems * (uint32_t)sizeof(ValT), bar, pol);
        }
    }
    if (tid < pr.tail_cnt) s_rend[pr.tail_beg - pr.a0 + tid] = __ldg(Ap + pr.tail_beg + tid);
    if (tid < pc.tail_cnt) {
        s_col[pc.tail_beg - pc.a0 + tid] = __ldg(Aj + pc.tail_beg + tid);
        s_val[pc.tail_beg - pc.a0 + tid] = __ldg(Ax + pc.tail_beg + tid);
    }
    const ValT alpha = alpha_dev ? __ldg(alpha_dev) : (ValT)1;
    const uint64_t pol_x = policy_evict_last();

    mbar_wait(bar, 0);
    __syncthreads();

    // ---- this thread's 8 consecutive slots: gather x (all loads issued before first use)
    const OffT *rend = s_rend + pr.shift;
    const int slot0 = tid * IPT;
    ValT p[IPT];
    {
        const int4 ca = *reinterpret_cast<const int4 *>(s_col + slot0);
        const int4 cb = *reinterpret_cast<const int4 *>(s_col + slot0 + 4);
        const int c[IPT] = {ca.x, ca.y, ca.z, ca.w, cb.x, cb.y, cb.z, cb.w};
        ValT xv[IPT];
#pragma unroll
        for (int k = 0; k < IPT; ++k) {
            const int i = slot0 + k - shift;  // tile-local nonzero index
            xv[k] = (i >= 0 && i < Z) ? ldg_hint(x + c[k], pol_x) : (ValT)0;
        }
        // ---- row-start flags: the nonzero at which row sx+j+1 begins, one thread per row end
        for (int j = tid; j < R; j += kMergeBlock) {
            const int64_t q = (int64_t)rend[j] - sy;
            if (q < Z) s_flag[(int)q + shift] = 1;
        }
        lds8(s_val + slot0, p);
#pragma unroll
        for (int k = 0; k < IPT; ++k) {
            const int i = slot0 + k - shift;
            p[k] = (i >= 0 && i < Z) ? p[k] * xv[k] : (ValT)0;
        }
    }
    __syncthreads();

    // ---- segmented scan.  pass 1: this thread's aggregate (saw a flag, sum since last flag)
    const uint2 fw = *reinterpret_cast<const uint2 *>(s_flag + slot0);
    const unsigned long long fbits = ((unsigned long long)fw.y << 32) | fw.x;  // byte k = flag k
    int flag = fbits != 0ull;
    ValT val = (ValT)0;
#pragma unroll
    for (int k = 0; k < IPT; ++k) val = ((fbits >> (8 * k)) & 1ull) ? p[k] : val + p[k];

    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const ValT pvv = __shfl_up_sync(0xffffffffu, val, d);
        const int pf = __shfl_up_sync(0xffffffffu, flag, d);
        if (lane >= d) {
            if (!flag) val += pvv;
            flag |= pf;
        }
    }
    if (lane == 31) {
        s_wval[warp] = val;
        s_wflag[warp] = flag;
    }
    ValT ev = __shfl_up_sync(0xffffffffu, val, 1);
    int ef = __shfl_up_sync(0xffffffffu, flag, 1);
    if (lane == 0) {
        ev = (ValT)0;
        ef = 0;
    }
    __syncthreads();
    ValT wv = (ValT)0;
#pragma unroll
    for (int w = 0; w < kMergeBlock / 32; ++w) {
        if (w < warp) {
            const ValT v = s_wval[w];
            wv = s_wflag[w] ? v : wv + v;
        }
    }
    // pass 2: running sums from the carry-in, written back over the products
    ValT run = ef ? ev : wv + ev;
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        run = ((fbits >> (8 * k)) & 1ull) ? p[k] : run + p[k];
        p[k] = run;
    }
    sts8(s_val + slot0, p);
    __syncthreads();

    // ---- one thread per row end: the row's total is the scan value at its last nonzero
    const ValT *scan = s_val + shift;
    for (int j = tid; j < R; j += kMergeBlock) {
        const int q = (int)((int64_t)rend[j] - sy);
        const int b = j > 0 ? (int)((int64_t)rend[j - 1] - sy) : 0;
        const ValT sum = q > b ? scan[q - 1] : (ValT)0;
        store_y_nonempty(y, peers, (int64_t)sx + j, alpha * sum, q > b);
    }
    if (tid == 0) {
        // nonzeros after the last row end of the tile belong to row ex: carry them out
        const int lastq = R > 0 ? (int)((int64_t)rend[R - 1] - sy) : 0;
        carry_row[tile] = ex;
        carry_val[tile] = Z > lastq ? scan[Z - 1] : (ValT)0;
    }
}

// ------------------------------------------------------------- tile kernel, register staging
// The default.  Same tile, same segmented scan, but Aj / Ax go from global memory straight
// into registers (two 128-bit loads each per thread, 32 contiguous bytes per lane) and the row
// ends are read by the thread that owns the row, so the only shared memory left is the scan
// array and the flags: 10 KB (fp32) or 18 KB (fp64) per CTA instead of 27-35 KB.
// Why it matters: the unified L1/shared array is what holds the lines of the x gathers that
// are in flight.  With the TMA-staged tile, 6 CTAs took 160-209 KB of it and left 20-68 KB of
// L1; ncu showed the gather rate tracking that remainder (o64: 35 KB/CTA -> 2.45 ms on R-MAT
// scale 24, o32: 27 KB/CTA -> 1.32 ms, all-shared carveout -> 2.4 ms), and at scale 27, where
// every miss is a DRAM round trip, the kernel ran at 7 % of the byte roofline.
template <typename ValT> struct LoadVals;
template <> struct LoadVals<float> {
    static __device__ __forceinline__ void vec8(const float *p, uint64_t pol, float (&v)[8]) {
        const float4 a = ldg_stream_val4(p, pol), b = ldg_stream_val4(p + 4, pol);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
        v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
};
template <> struct LoadVals<double> {
    static __device__ __forceinline__ void vec8(const double *p, uint64_t pol, double (&v)[8]) {
        const double4_t a = ldg_stream_val4(p, pol), b = ldg_stream_val4(p + 4, pol);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
        v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
};

// a warp's total for the cross-warp fold: (sum since its last row start, that row / a flag)
template <typename ValT> struct WarpTotal;
template <> struct __align__(8) WarpTotal<float> { float val; int rid; };
template <> struct __align__(16) WarpTotal<double> { double val; int rid; int pad; };

// HOT: Aj is the remapped copy of a hot-x plan (hotx.cu): an index with the top bit set is a rank
// into the dense copy of the hot columns' x; x_hot_biased = x_hot - 2^31 elements, so that either
// base + (uint32) index is the address.
// The shared memory of one tile in flight.
template <int BLOCK, typename ValT>
struct __align__(16) TileSmem {
    ValT scan[BLOCK * kMergeIPT];
    WarpTotal<ValT> w[BLOCK / 32];
};

// Tile descriptors of the persistent kernel, built once per partition by tile_desc_kernel:
//   row_end[r]  = Ap[r+1] - sy(t), t the tile in which row r's end item lies (<= TILE: 16 bits);
//   start_mask  = 1 bit per slot and tile, bit s of tile t set iff a row starts at slot s -- the
//                 byte flags that the scatter of Ap writes in the GROUPS == 1 body.
struct TileDesc {
    const uint16_t *row_end;
    const unsigned char *start_mask;
};
// Only the persistent fp32 kernel with 64-bit offsets uses them: there they are about half the bytes of
// Ap (2 B per row + 128 B per tile against 8 B per row; R-MAT scale 27: 0.55 against 1.07 GB per
// SpMV).  With 32-bit offsets they are as many bytes as Ap, and the kernel that used them (and its
// coordinates one tile ahead) measured slower: R-MAT scale 24, static pattern, 994 -> 1031 us per SpMV.
// descriptor loads: read once per SpMV, so they bypass the L1 and go first out of the L2, where they
// would otherwise push out lines of x (R-MAT scale 27: step 10.78 with plain loads, 10.62 ms with these)
__device__ __forceinline__ unsigned ldg_stream_u8(const unsigned char *p, uint64_t policy) {
    unsigned v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u8 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(policy));
    return v;
}
__device__ __forceinline__ int ldg_stream_u16(const uint16_t *p, uint64_t policy) {
    unsigned v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u16 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(policy));
    return (int)v;
}
// fp64 (off by default in the table kernel) keeps Ap as well: its body spills with the descriptors.
template <int GROUPS, typename OffT, typename ValT> constexpr bool tile_desc_used() {
    return GROUPS > 1 && sizeof(OffT) == 8 && sizeof(ValT) == 4;
}

// GROUPS == 1: the CTA is one tile (tile = blockIdx.x, static shared memory, __syncthreads).
// GROUPS > 1 (merge_tile_table_kernel): the CTA is GROUPS independent groups of BLOCK threads, each
// working on its own tile out of its own TileSmem and flags with its own named barrier, and `table`
// holds the x values of ranks 0 .. table_n-1 of the hot-x plan in shared memory.
// DESC (tile_desc_used): the caller passes the tile's coordinates (sx, ex), and the row ends and row
// starts come from the tile descriptors: no load of Ap, no flags, no flag scatter and two barriers
// per tile instead of four.  Otherwise the row ends come from Ap.
template <int BLOCK, int HAS_PEERS, bool HOT, int GROUPS, typename OffT, typename ValT>
__device__ __forceinline__ void
merge_tile_reg_body(int32_t n_rows, OffT nnz, const OffT *__restrict__ Ap,
                    const int32_t *__restrict__ Aj, const ValT *__restrict__ Ax,
                    const ValT *__restrict__ x, ValT *__restrict__ y,
                    const ValT *__restrict__ alpha_dev, const PeerOut &peers,
                    const int32_t *__restrict__ coords_x, int32_t *__restrict__ carry_row,
                    ValT *__restrict__ carry_val, const ValT *__restrict__ x_hot_biased,
                    int64_t tile_of_group = 0, TileSmem<BLOCK, ValT> *group_smem = nullptr,
                    const ValT *table = nullptr, uint32_t table_n = 0, unsigned char *group_flag = nullptr,
                    int32_t group_sx = 0, int32_t group_ex = 0, TileDesc desc = {}) {
    constexpr int IPT = kMergeIPT;
    constexpr int SLOTS = BLOCK * IPT;
    constexpr int TILE = SLOTS - 4;  // path items per tile
    constexpr bool DESC = tile_desc_used<GROUPS, OffT, ValT>();
    TileSmem<BLOCK, ValT> *sm = group_smem;
    unsigned char *s_flag = group_flag;
    if constexpr (GROUPS == 1) {
        __shared__ TileSmem<BLOCK, ValT> s_cta;
        // row-start flags, one byte per slot.  (One BIT per slot, set with atomicOr, saves 1.8 KB per
        // 256-thread CTA and fits one more CTA per SM inside the 64 KB carveout, but measured slower:
        // R-MAT scale 24 1146 -> 1166 us, scale 27 14.70 -> 14.93 ms.)
        __shared__ __align__(16) unsigned char s_cta_flag[SLOTS];
        sm = &s_cta;
        s_flag = s_cta_flag;
    }
    ValT *const s_scan = sm->scan;
    WarpTotal<ValT> *const s_w = sm->w;
    const int grp = GROUPS == 1 ? 0 : (int)(threadIdx.x / BLOCK);
    auto tile_sync = [grp]() {
        if (GROUPS == 1) __syncthreads();
        else asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "n"(BLOCK) : "memory");
    };

    const int tid = GROUPS == 1 ? (int)threadIdx.x : (int)(threadIdx.x % BLOCK);
    const int64_t tile = GROUPS == 1 ? (int64_t)blockIdx.x : tile_of_group;
    const int64_t total = (int64_t)n_rows + (int64_t)nnz;
    const int64_t d0 = tile * TILE;
    const int64_t d1 = d0 + TILE < total ? d0 + TILE : total;
    const int32_t sx = DESC ? group_sx : __ldg(coords_x + tile);
    const int32_t ex = DESC ? group_ex : __ldg(coords_x + tile + 1);
    const int64_t sy = d0 - sx;
    const int R = ex - sx;                // rows that end inside this tile
    const int Z = (int)((d1 - ex) - sy);  // nonzeros inside this tile
    const int shift = (int)(sy & 3);      // slot s holds tile-local nonzero s - shift
    const int64_t a0 = sy - shift;        // 16-byte aligned position of slot 0 in Aj / Ax

    if constexpr (!DESC) *reinterpret_cast<uint2 *>(s_flag + tid * IPT) = make_uint2(0u, 0u);

    // ---- DESC: this thread's byte of the start mask (its 8 slots' row-start bits), and the
    // row ends of its first row (q0) and of the row before (b0), issued with the Aj / Ax loads so that
    // they have arrived when the scan ends.  Row sx's nonzeros start at or before sy (the merge path
    // has Ap[sx] <= sy), hence b = 0 for j = 0.
    unsigned mask_byte = 0;
    int q0 = 0, b0 = 0;
    if constexpr (DESC) {
        const uint64_t pol_desc = policy_evict_first();
        mask_byte = ldg_stream_u8(desc.start_mask + tile * (SLOTS / 8) + tid, pol_desc);
        if (tid < R) q0 = ldg_stream_u16(desc.row_end + sx + tid, pol_desc);
        // lanes 1..31 take b0 from the lane below after the gathers; lane 0 loads its own
        if ((tid & 31) == 0 && tid > 0 && tid < R) b0 = ldg_stream_u16(desc.row_end + sx + tid - 1, pol_desc);
    }

    // ---- this thread's 8 consecutive slots straight into registers
    const int slot0 = tid * IPT;
    const uint64_t pol_stream = policy_evict_first();
    const uint64_t pol_x = policy_evict_last();
    int c[IPT];
    ValT p[IPT];
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        c[k] = 0;
        p[k] = (ValT)0;
    }
    if (slot0 < shift + Z) {
        const int64_t g = a0 + slot0;
        if (g + IPT <= (int64_t)nnz) {
            const int4 ca = ldg_stream_int4(Aj + g, pol_stream);
            const int4 cb = ldg_stream_int4(Aj + g + 4, pol_stream);
            c[0] = ca.x; c[1] = ca.y; c[2] = ca.z; c[3] = ca.w;
            c[4] = cb.x; c[5] = cb.y; c[6] = cb.z; c[7] = cb.w;
            LoadVals<ValT>::vec8(Ax + g, pol_stream, p);
        } else {  // the last vectors of the matrix: element-wise, inside the arrays
#pragma unroll
            for (int k = 0; k < IPT; ++k) {
                if (g + k < (int64_t)nnz) {
                    c[k] = __ldg(Aj + g + k);
                    p[k] = __ldg(Ax + g + k);
                }
            }
        }
    }
    const ValT alpha = alpha_dev ? __ldg(alpha_dev) : (ValT)1;
    if constexpr (!DESC) {
        tile_sync();  // flags are clear
        // ---- row-start flags, one thread per row end (Ap read coalesced, no staging)
        for (int j = tid; j < R; j += BLOCK) {
            const int64_t q = (int64_t)__ldg(Ap + sx + 1 + j) - sy;
            if (q < Z) s_flag[(int)q + shift] = 1;
        }
    }
    // ---- x gathers, all eight issued before the first use
    {
        ValT xv[IPT];
#pragma unroll
        for (int k = 0; k < IPT; ++k) {
            const int i = slot0 + k - shift;
            const ValT *src = HOT ? (c[k] < 0 ? x_hot_biased : x) + (uint32_t)c[k] : x + c[k];
            if (GROUPS > 1) {
                // rank of a hot column, >= 2^31 for any other: one compare picks the table
                const uint32_t r = (uint32_t)c[k] ^ 0x80000000u;
                if (i >= 0 && i < Z) xv[k] = r < table_n ? table[r] : ldg_hint(src, pol_x);
                else xv[k] = (ValT)0;
            } else {
                xv[k] = (i >= 0 && i < Z) ? ldg_hint(src, pol_x) : (ValT)0;
            }
        }
#pragma unroll
        for (int k = 0; k < IPT; ++k) {
            const int i = slot0 + k - shift;
            p[k] = (i >= 0 && i < Z) ? p[k] * xv[k] : (ValT)0;
        }
    }
    if constexpr (DESC) {   // the row end before this thread's first row: the lane below's q0
        const int up = __shfl_up_sync(0xffffffffu, q0, 1);
        if ((tid & 31) != 0) b0 = up;
    }
    // ---- segmented scan (as in the TMA variant).  The flag of slot k is bit FS * k of fbits: the
    // bytes of the shared flags or the bits of the start mask (DESC).
    constexpr int FS = DESC ? 1 : 8;
    unsigned long long fbits = mask_byte;
    if constexpr (!DESC) {
        tile_sync();  // flags are set
        const uint2 fw = *reinterpret_cast<const uint2 *>(s_flag + slot0);
        fbits = ((unsigned long long)fw.y << 32) | fw.x;
    }
    int flag = fbits != 0ull;
    ValT val = (ValT)0;
#pragma unroll
    for (int k = 0; k < IPT; ++k) val = ((fbits >> (FS * k)) & 1ull) ? p[k] : val + p[k];
    const int lane = tid & 31, warp = tid >> 5;
    // the row-start bits of the warp as one ballot: lane L's sum reaches back to lane L - d iff
    // none of lanes L - d + 1 .. L holds a flag -- 6 shuffles per thread instead of 12
    const unsigned fmask = __ballot_sync(0xffffffffu, flag != 0);
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const ValT pvv = __shfl_up_sync(0xffffffffu, val, d);
        if (lane >= d && ((fmask >> (lane - d + 1)) & ((1u << d) - 1u)) == 0u) val += pvv;
    }
    if (lane == 31) {   // (sum since the warp's last flag, any flag): one shared-memory word
        s_w[warp].val = val;
        s_w[warp].rid = fmask != 0u;
    }
    ValT ev = __shfl_up_sync(0xffffffffu, val, 1);
    if (lane == 0) ev = (ValT)0;
    const bool ef = (fmask & ((1u << lane) - 1u)) != 0u;
    tile_sync();
    ValT wv = (ValT)0;
#pragma unroll
    for (int w = 0; w < BLOCK / 32; ++w) {
        if (w < warp) {
            const WarpTotal<ValT> t = s_w[w];
            wv = t.rid ? t.val : wv + t.val;
        }
    }
    ValT run = ef ? ev : wv + ev;
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        run = ((fbits >> (FS * k)) & 1ull) ? p[k] : run + p[k];
        p[k] = run;
    }
    sts8(s_scan + slot0, p);
    tile_sync();

    // ---- one thread per row end: the row's total is the scan value at its last nonzero.
    // Row sx+j covers tile-local nonzeros [max(Ap[sx+j]-sy, 0), Ap[sx+j+1]-sy).
    const ValT *scan = s_scan + shift;
    for (int j = tid; j < R; j += BLOCK) {
        int q, b;
        if constexpr (!DESC) {
            const int64_t b64 = (int64_t)__ldg(Ap + sx + j) - sy;
            q = (int)((int64_t)__ldg(Ap + sx + 1 + j) - sy);
            b = b64 > 0 ? (int)b64 : 0;
        } else if (j == tid) {
            q = q0;
            b = b0;
        } else {  // more than BLOCK rows end in the tile (runs of empty rows)
            q = __ldg(desc.row_end + sx + j);
            b = __ldg(desc.row_end + sx + j - 1);
        }
        const ValT sum = q > b ? scan[q - 1] : (ValT)0;
        // the peer fan-out is compiled in only when there are peers: its code cost the
        // (o32, fp32) kernel its 32-register budget (spills; c3 1224 -> 1459 us)
        // HAS_PEERS 2: the peers are one NVLink multicast address -- a single pointer instead of the
        // list keeps the kernel inside 32 registers (the list costs 8 more and two CTAs per SM)
        if (HAS_PEERS == 2) {
            y[(int64_t)sx + j] = alpha * sum;
            if (q > b) multimem_st(static_cast<ValT *>(peers.ptr[0]) + (int64_t)sx + j, alpha * sum);
        } else if (HAS_PEERS) {
            store_y_nonempty(y, peers, (int64_t)sx + j, alpha * sum, q > b);
        } else {
            y[(int64_t)sx + j] = alpha * sum;
        }
        if (DESC && j == R - 1) {  // the tile's last row end is in hand: carry out what follows it
            carry_row[tile] = ex;
            carry_val[tile] = Z > q ? scan[Z - 1] : (ValT)0;
        }
    }
    if (tid == 0 && (!DESC || R == 0)) {
        // nonzeros after the last row end of the tile belong to row ex: carry them out
        const int64_t lq = !DESC && R > 0 ? (int64_t)__ldg(Ap + ex) - sy : 0;
        const int lastq = lq > 0 ? (int)lq : 0;
        carry_row[tile] = ex;
        carry_val[tile] = Z > lastq ? scan[Z - 1] : (ValT)0;
    }
}

// ------------------------------------------------------------- tile kernel, marker form
// Same tile, same loads, same products as merge_tile_reg_body, but the rows are delimited by a
// 16-bit MARKER per slot -- the number (relative to the tile's first row, plus one) of the row
// that starts there -- instead of a byte flag.  The segmented scan then carries the row number
// along with the running sum, and a thread that walks over a marker knows which row has just
// ended and with what total: it drops it into s_y[row] there and then.  What this removes from
// the flag form (profiles/r1_merge_c5_v4: short_scoreboard + mio_throttle + barrier cost more
// issue time than the memory latency):
//   * the scan values are never written back to shared memory (two 128-bit stores per thread),
//     and nobody reads Ap a second time to pick a row's total out of them;
//   * the row-start bits of a warp travel as one ballot, so the shuffle scan moves 6 values per
//     thread instead of 12;
//   * (value, row) of a warp's total is one 8-byte shared-memory word: half the loads of the
//     cross-warp fold;
//   * the rows a warp completes are consecutive, so the warp stores them itself after a
//     __syncwarp: three CTA barriers per tile instead of four.
// Row r of the tile is written to y by exactly one thread: the one that holds the marker of the
// next non-empty row (its total), or -- if r has no nonzeros at all -- the thread that set the
// markers (0).  Summation order inside a row is unchanged (thread-serial, then lanes, then warps).

template <int BLOCK, int HAS_PEERS, bool HOT, typename OffT, typename ValT>
__device__ __forceinline__ void
merge_tile_mark_body(int32_t n_rows, OffT nnz, const OffT *__restrict__ Ap,
                     const int32_t *__restrict__ Aj, const ValT *__restrict__ Ax,
                     const ValT *__restrict__ x, ValT *__restrict__ y,
                     const ValT *__restrict__ alpha_dev, const PeerOut &peers,
                     const int32_t *__restrict__ coords_x, int32_t *__restrict__ carry_row,
                     ValT *__restrict__ carry_val, const ValT *__restrict__ x_hot_biased) {
    constexpr int IPT = kMergeIPT;
    constexpr int SLOTS = BLOCK * IPT;
    constexpr int TILE = SLOTS - 4;
    static_assert(TILE < 65535, "row numbers are 16-bit markers");
    __shared__ __align__(16) ValT s_y[SLOTS];                // totals of the rows that end in the tile
    __shared__ __align__(16) unsigned short s_mark[SLOTS];   // slot -> 1 + row starting there, 0 = none
    __shared__ WarpTotal<ValT> s_w[BLOCK / 32];

    const int tid = threadIdx.x;
    const int64_t tile = blockIdx.x;
    const int64_t total = (int64_t)n_rows + (int64_t)nnz;
    const int64_t d0 = tile * TILE;
    const int64_t d1 = d0 + TILE < total ? d0 + TILE : total;
    const int32_t sx = __ldg(coords_x + tile);
    const int32_t ex = __ldg(coords_x + tile + 1);
    const int64_t sy = d0 - sx;
    const int R = ex - sx;
    const int Z = (int)((d1 - ex) - sy);
    const int shift = (int)(sy & 3);
    const int64_t a0 = sy - shift;

    *reinterpret_cast<uint4 *>(s_mark + tid * IPT) = make_uint4(0u, 0u, 0u, 0u);

    const int slot0 = tid * IPT;
    const uint64_t pol_stream = policy_evict_first();
    const uint64_t pol_x = policy_evict_last();
    int c[IPT];
    ValT p[IPT];
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        c[k] = 0;
        p[k] = (ValT)0;
    }
    if (slot0 < shift + Z) {
        const int64_t g = a0 + slot0;
        if (g + IPT <= (int64_t)nnz) {
            const int4 ca = ldg_stream_int4(Aj + g, pol_stream);
            const int4 cb = ldg_stream_int4(Aj + g + 4, pol_stream);
            c[0] = ca.x; c[1] = ca.y; c[2] = ca.z; c[3] = ca.w;
            c[4] = cb.x; c[5] = cb.y; c[6] = cb.z; c[7] = cb.w;
            LoadVals<ValT>::vec8(Ax + g, pol_stream, p);
        } else {
#pragma unroll
            for (int k = 0; k < IPT; ++k) {
                if (g + k < (int64_t)nnz) {
                    c[k] = __ldg(Aj + g + k);
                    p[k] = __ldg(Ax + g + k);
                }
            }
        }
    }
    const ValT alpha = alpha_dev ? __ldg(alpha_dev) : (ValT)1;
    __syncthreads();  // markers are clear

    // ---- markers, one thread per row end j (row sx+j ends, row sx+j+1 starts at q).  Of a run of
    // rows starting at the same position only the last has nonzeros from there on: it sets the
    // marker; a row without nonzeros is finished here (0).
    for (int j = tid; j < R; j += BLOCK) {
        const OffT b = __ldg(Ap + sx + j);
        const OffT e = __ldg(Ap + sx + 1 + j);
        const int q = (int)((int64_t)e - sy);
        if (j == R - 1 || __ldg(Ap + sx + 2 + j) != e) s_mark[q + shift] = (unsigned short)(j + 1);
        if (b == e) s_y[j] = (ValT)0;
    }
    // ---- x gathers, all eight issued before the first use
    {
        ValT xv[IPT];
#pragma unroll
        for (int k = 0; k < IPT; ++k) {
            const int i = slot0 + k - shift;
            const ValT *src = HOT ? (c[k] < 0 ? x_hot_biased : x) + (uint32_t)c[k] : x + c[k];
            xv[k] = (i >= 0 && i < Z) ? ldg_hint(src, pol_x) : (ValT)0;
        }
#pragma unroll
        for (int k = 0; k < IPT; ++k) {
            const int i = slot0 + k - shift;
            p[k] = (i >= 0 && i < Z) ? p[k] * xv[k] : (ValT)0;
        }
    }
    __syncthreads();  // markers are set

    // ---- this thread's eight markers; pass 1: (sum since the last marker, last row started)
    const uint4 mw = *reinterpret_cast<const uint4 *>(s_mark + slot0);
    const unsigned m32[4] = {mw.x, mw.y, mw.z, mw.w};
    int mk[IPT];
#pragma unroll
    for (int k = 0; k < IPT; ++k) mk[k] = (int)((m32[k >> 1] >> (16 * (k & 1))) & 0xffffu);
    ValT val = (ValT)0;
    int rid = 0;
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        val = mk[k] ? p[k] : val + p[k];
        rid = mk[k] ? mk[k] : rid;
    }
    const int lane = tid & 31, warp = tid >> 5;
    // lanes holding a marker, as one word: lane L's sum extends back to lane L - d iff none of
    // lanes L - d + 1 .. L holds one
    const unsigned fmask = __ballot_sync(0xffffffffu, rid != 0);
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const ValT pv = __shfl_up_sync(0xffffffffu, val, d);
        if (lane >= d && ((fmask >> (lane - d + 1)) & ((1u << d) - 1u)) == 0u) val += pv;
    }
    // carry into this lane from the lanes below it: their inclusive sum, and the row they are in
    ValT ev = __shfl_up_sync(0xffffffffu, val, 1);
    if (lane == 0) ev = (ValT)0;
    const unsigned below = fmask & ((1u << lane) - 1u);
    const int src_lane = below ? 31 - __clz(below) : 0;
    int erow = __shfl_sync(0xffffffffu, rid, src_lane);
    if (lane == 31) {   // the warp's total: sum since its last marker, and that marker's row (0 = none)
        s_w[warp].val = val;
        s_w[warp].rid = rid ? rid : (below ? erow : 0);
    }
    __syncthreads();
    ValT wv = (ValT)0;
    int wrow = 0;
#pragma unroll
    for (int w = 0; w < BLOCK / 32; ++w) {
        if (w < warp) {
            const WarpTotal<ValT> t = s_w[w];
            wv = t.rid ? t.val : wv + t.val;
            wrow = t.rid ? t.rid : wrow;
        }
    }
    // ---- pass 2: walk the slots again from the carry-in; a marker closes the current row
    ValT run = below ? ev : wv + ev;
    int row = below ? erow : wrow;
    const int first_row = row;
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        if (mk[k]) {
            s_y[row] = alpha * run;
            run = p[k];
            row = mk[k];
        } else {
            run += p[k];
        }
    }
    // ---- the rows this warp completed are consecutive: [row entering lane 0, row leaving lane 31)
    __syncwarp();
    const int r_begin = __shfl_sync(0xffffffffu, first_row, 0);
    const int r_end = __shfl_sync(0xffffffffu, row, 31);
    for (int j = r_begin + lane; j < r_end; j += 32) {
        const ValT v = s_y[j];
        if (HAS_PEERS) {
            // peers only get rows with nonzeros in this tile (see store_y_nonempty)
            const int64_t b64 = (int64_t)__ldg(Ap + sx + j) - sy;
            const int64_t q64 = (int64_t)__ldg(Ap + sx + 1 + j) - sy;
            const bool has = q64 > (b64 > 0 ? b64 : 0);
            if (HAS_PEERS == 2) {
                y[(int64_t)sx + j] = v;
                if (has) multimem_st(static_cast<ValT *>(peers.ptr[0]) + (int64_t)sx + j, v);
            } else {
                store_y_nonempty(y, peers, (int64_t)sx + j, v, has);
            }
        } else {
            y[(int64_t)sx + j] = v;
        }
    }
    if (tid == BLOCK - 1) {
        // what follows the last row end belongs to row ex: carry it out
        carry_row[tile] = sx + row;
        carry_val[tile] = run;
    }
}

// Two entry points over one body, because the register budget is set per __global__: with
// 32-bit offsets and fp32 the body fits 32 registers without spilling (8 CTAs/SM; c3 1328 ->
// 1230 us); the 64-bit-offset and fp64 bodies spill under that cap and are left to ptxas
// (40 / 64 registers, 6 / 4 CTAs per SM).
#define MERGE_REG_KERNEL_ARGS                                                                    \
    int32_t n_rows, OffT nnz, const OffT *__restrict__ Ap, const int32_t *__restrict__ Aj,       \
    const ValT *__restrict__ Ax, const ValT *__restrict__ x, ValT *__restrict__ y,               \
    const ValT *__restrict__ alpha_dev, PeerOut peers, const int32_t *__restrict__ coords_x,     \
    int32_t *__restrict__ carry_row, ValT *__restrict__ carry_val
// ALGO 0 = marker form (the default), 1 = the flag form of round 1 (option "merge_algo", A/B)
template <int ALGO, int BLOCK, int HAS_PEERS, bool HOT, typename OffT, typename ValT>
__device__ __forceinline__ void merge_tile_dispatch(MERGE_REG_KERNEL_ARGS, const ValT *__restrict__ x_hot_biased) {
    if (ALGO == 0)
        merge_tile_mark_body<BLOCK, HAS_PEERS, HOT, OffT, ValT>(n_rows, nnz, Ap, Aj, Ax, x, y, alpha_dev, peers,
                                                                coords_x, carry_row, carry_val, x_hot_biased);
    else
        merge_tile_reg_body<BLOCK, HAS_PEERS, HOT, 1, OffT, ValT>(n_rows, nnz, Ap, Aj, Ax, x, y, alpha_dev, peers,
                                                               coords_x, carry_row, carry_val, x_hot_biased);
}
template <int ALGO, int BLOCK, int HAS_PEERS, typename OffT, typename ValT>
__global__ void __launch_bounds__(BLOCK, 2048 / BLOCK) merge_tile_reg_kernel_occ8(MERGE_REG_KERNEL_ARGS) {
    merge_tile_dispatch<ALGO, BLOCK, HAS_PEERS, false, OffT, ValT>(n_rows, nnz, Ap, Aj, Ax, x, y, alpha_dev, peers,
                                                                   coords_x, carry_row, carry_val, nullptr);
}
template <int ALGO, int BLOCK, int HAS_PEERS, typename OffT, typename ValT>
__global__ void __launch_bounds__(BLOCK) merge_tile_reg_kernel(MERGE_REG_KERNEL_ARGS) {
    merge_tile_dispatch<ALGO, BLOCK, HAS_PEERS, false, OffT, ValT>(n_rows, nnz, Ap, Aj, Ax, x, y, alpha_dev, peers,
                                                                   coords_x, carry_row, carry_val, nullptr);
}
// the hot-x variant: Aj is the plan's remapped copy
template <int ALGO, int BLOCK, int HAS_PEERS, typename OffT, typename ValT>
__global__ void __launch_bounds__(BLOCK, 2048 / BLOCK)
merge_tile_hot_kernel_occ8(MERGE_REG_KERNEL_ARGS, const ValT *__restrict__ x_hot_biased) {
    merge_tile_dispatch<ALGO, BLOCK, HAS_PEERS, true, OffT, ValT>(n_rows, nnz, Ap, Aj, Ax, x, y, alpha_dev, peers,
                                                                  coords_x, carry_row, carry_val, x_hot_biased);
}
template <int ALGO, int BLOCK, int HAS_PEERS, typename OffT, typename ValT>
__global__ void __launch_bounds__(BLOCK)
merge_tile_hot_kernel(MERGE_REG_KERNEL_ARGS, const ValT *__restrict__ x_hot_biased) {
    merge_tile_dispatch<ALGO, BLOCK, HAS_PEERS, true, OffT, ValT>(n_rows, nnz, Ap, Aj, Ax, x, y, alpha_dev, peers,
                                                                  coords_x, carry_row, carry_val, x_hot_biased);
}
// The persistent form of the hot-x tile kernel: one CTA per SM, kTableGroups groups of 128 threads
// that each walk over tiles (tile = round * gridDim.x * groups + blockIdx.x * groups + group: at
// any moment the SMs work on neighbouring tiles, as a plain launch would), so that shared memory
// can hold a TABLE: the x values of the plan's first table_n ranks, its most frequent columns.
// Why: ncu puts the flag-form kernel on R-MAT scale 24 at 86 % of l1tex__m_l1tex2xbar_req_cycles --
// one request per cycle per SM from the L1 to the L2 is the wall every CSR kernel here runs into
// (~270 G gathers/s on the chip, tools/l2_gather_probe.cu), and only 7 % of the gathers hit the
// L1.  A gather served from shared memory never becomes such a request.
// Measured (tools/table_sweep.py, L2 flushed, y bit-identical in every row):
//   scale 24 (x 64 MB, all-table plan): 1100 us plain -> 1105 persistent without a table -> 1000
//     with 31 K columns (36 % of the gathers) in the table; with 13 K columns request cycles go
//     from 86 to 73 % and the kernel is then short of warps (8 per scheduler at 56 registers; two
//     or three smaller CTAs per SM, each with its own table, were slower: 1070 / 1175 / 1367 us);
//   scale 27 (hot-x plan + table): 11.4 ms -> 10.9 persistent -> 10.4 with 15 K columns (15 %).
// The table takes its space from the L1, which is what holds the gathers in flight; the sizes
// are chosen in launch_merge ("hot_x_table_bytes").  The tile body is the flag form's, with
// group-local barriers; products and their order are unchanged.  The partition is fixed while the
// kernel is reused, so with 64-bit offsets and fp32 its row ends and row starts are read from tile
// descriptors built once with it (TileDesc) instead of from Ap, and each group loads its next
// tile's coordinates a tile ahead.
#ifndef SPMV_TABLE_GROUPS
#define SPMV_TABLE_GROUPS 8
#endif
constexpr int kTableGroups = SPMV_TABLE_GROUPS;
#ifndef SPMV_TABLE_CTAS
#define SPMV_TABLE_CTAS 1
#endif
constexpr int kTableCtas = SPMV_TABLE_CTAS;   // CTAs per SM, each with its own copy of the table
constexpr int kTableBlock = 128;
template <int HAS_PEERS, typename OffT, typename ValT>
__global__ void __launch_bounds__(kTableGroups *kTableBlock, kTableCtas)
merge_tile_table_kernel(MERGE_REG_KERNEL_ARGS, const ValT *__restrict__ x_hot_biased,
                        const ValT *__restrict__ x_hot, uint32_t table_n, int64_t num_tiles, TileDesc desc) {
    constexpr bool DESC = tile_desc_used<kTableGroups, OffT, ValT>();
    extern __shared__ __align__(128) unsigned char smem_raw[];
    using Smem = TileSmem<kTableBlock, ValT>;
    Smem *const groups = reinterpret_cast<Smem *>(smem_raw);
    unsigned char *const flags = smem_raw + sizeof(Smem) * kTableGroups;   // without descriptors
    ValT *const table = reinterpret_cast<ValT *>(flags + (DESC ? 0 : kTableGroups * kTableBlock * kMergeIPT));
    for (uint32_t i = threadIdx.x; i < table_n; i += kTableGroups * kTableBlock) table[i] = __ldg(x_hot + i);
    __syncthreads();
    const int grp = (int)(threadIdx.x / kTableBlock);
    unsigned char *const group_flag = DESC ? nullptr : flags + grp * kTableBlock * kMergeIPT;
    const int64_t stride = (int64_t)gridDim.x * kTableGroups;
    int64_t tile = (int64_t)blockIdx.x * kTableGroups + grp;
    int32_t sx = 0, ex = 0;
    if (DESC && tile < num_tiles) {
        sx = __ldg(coords_x + tile);
        ex = __ldg(coords_x + tile + 1);
    }
    for (; tile < num_tiles; tile += stride) {
        // DESC: the group's next tile's coordinates, one tile ahead -- every other load of a tile
        // depends on them
        int32_t next_sx = 0, next_ex = 0;
        if (DESC && tile + stride < num_tiles) {
            next_sx = __ldg(coords_x + tile + stride);
            next_ex = __ldg(coords_x + tile + stride + 1);
        }
        merge_tile_reg_body<kTableBlock, HAS_PEERS, true, kTableGroups, OffT, ValT>(
            n_rows, nnz, Ap, Aj, Ax, x, y, alpha_dev, peers, coords_x, carry_row, carry_val, x_hot_biased, tile,
            groups + grp, table, table_n, group_flag, sx, ex, desc);
        sx = next_sx;
        ex = next_ex;
    }
}
#undef MERGE_REG_KERNEL_ARGS

// The tile descriptors (TileDesc) of a partition, one thread per row: the tile in which row r's end
// item lies is (r + Ap[r+1]) / tile_items (the merge path puts it at diagonal r + Ap[r+1]).  The
// start mask must be zero on entry.
template <typename OffT>
__global__ void __launch_bounds__(256)
tile_desc_kernel(int32_t n_rows, OffT nnz, const OffT *__restrict__ Ap, const int32_t *__restrict__ coords_x,
                 uint16_t *__restrict__ row_end, uint32_t *__restrict__ start_mask) {
    constexpr int SLOTS = kTableBlock * kMergeIPT;
    constexpr int TILE = SLOTS - 4;
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const int64_t total = (int64_t)n_rows + (int64_t)nnz;
    const int64_t e = (int64_t)__ldg(Ap + r + 1);
    const int64_t t = (r + e) / TILE;
    const int64_t d0 = t * TILE;
    const int64_t d1 = d0 + TILE < total ? d0 + TILE : total;
    const int64_t sy = d0 - __ldg(coords_x + t);
    const int64_t ey = d1 - __ldg(coords_x + t + 1);
    const int q = (int)(e - sy);
    row_end[r] = (uint16_t)q;
    // row r+1 starts inside the tile (q < Z): slot q + shift, as the flag scatter sets it
    if (e < ey) {
        const int s = q + (int)(sy & 3);
        atomicOr(start_mask + t * (SLOTS / 32) + (s >> 5), 1u << (s & 31));
    }
}

// ------------------------------------------------------------------------- carry fixup
// One thread per tile.  Consecutive tiles whose carry lands in the same row form a run; the
// head of the run adds the run's carries, in tile order, to y[row].
template <typename ValT>
__global__ void __launch_bounds__(256)
merge_fixup_kernel(int32_t n_rows, int64_t num_tiles, const int32_t *__restrict__ carry_row,
                   const ValT *__restrict__ carry_val, ValT *__restrict__ y,
                   const ValT *__restrict__ alpha_dev, PeerOut peers) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= num_tiles) return;
    const int32_t row = carry_row[t];
    if (row >= n_rows) return;
    if (t > 0 && carry_row[t - 1] == row) return;
    ValT sum = carry_val[t];
    // a hub row spans hundreds of tiles: walk its run eight tiles at a time so that the loads
    // of a batch are in flight together (one load per trip made this kernel as long as the
    // search: 73 us on R-MAT scale 27); the additions stay in tile order
    bool more = true;
    for (int64_t u = t + 1; more && u < num_tiles; u += 8) {
        int32_t r[8];
        ValT v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const bool in = u + j < num_tiles;
            r[j] = in ? carry_row[u + j] : -1;
            v[j] = in ? carry_val[u + j] : (ValT)0;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            more = more && r[j] == row;
            if (more) sum += v[j];
        }
    }
    const ValT alpha = alpha_dev ? __ldg(alpha_dev) : (ValT)1;
    store_y(y, peers, (int64_t)row, y[row] + alpha * sum);
}

// ----------------------------------------------------- generalised (semiring) tile kernel
// y[r] = REDUCE_k COMBINE(Ax[k], x[Aj[k]]) starting from IDENTITY, the capability of the
// reference's SpMV_merge_based_generalized (merge_genl/merge_genl.cuh:19-38 with its
// functor_t{initialize, combine, reduce}; CPU twin cpu_navie.hpp:20-35).  A template functor
// cannot cross a C ABI, so the menu is fixed (SPMVB200_SEMIRING_*).  Same tile algorithm as
// merge_tile_reg_body; kept separate so the plus-times hot path is not perturbed.  With
// plus-times this kernel also serves y = alpha*A*x + beta*y.
template <typename ValT> struct SrPlusTimes {
    static constexpr bool kLinear = true;
    static __device__ __forceinline__ ValT identity() { return (ValT)0; }
    static __device__ __forceinline__ ValT combine(ValT a, ValT x) { return a * x; }
    static __device__ __forceinline__ ValT reduce(ValT u, ValT v) { return u + v; }
};
template <typename ValT> struct SrMinPlus {
    static constexpr bool kLinear = false;
    static __device__ __forceinline__ ValT identity() { return (ValT)INFINITY; }
    static __device__ __forceinline__ ValT combine(ValT a, ValT x) { return a + x; }
    static __device__ __forceinline__ ValT reduce(ValT u, ValT v) { return u < v ? u : v; }
};
template <typename ValT> struct SrMaxPlus {
    static constexpr bool kLinear = false;
    static __device__ __forceinline__ ValT identity() { return (ValT)-INFINITY; }
    static __device__ __forceinline__ ValT combine(ValT a, ValT x) { return a + x; }
    static __device__ __forceinline__ ValT reduce(ValT u, ValT v) { return u > v ? u : v; }
};
template <typename ValT> struct SrOrAnd {
    static constexpr bool kLinear = false;
    static __device__ __forceinline__ ValT identity() { return (ValT)0; }
    static __device__ __forceinline__ ValT combine(ValT a, ValT x) {
        return (a != (ValT)0 && x != (ValT)0) ? (ValT)1 : (ValT)0;
    }
    static __device__ __forceinline__ ValT reduce(ValT u, ValT v) { return u > v ? u : v; }
};

template <typename S, typename OffT, typename ValT>
__global__ void __launch_bounds__(kMergeBlock)
merge_tile_genl_kernel(int32_t n_rows, OffT nnz, const OffT *__restrict__ Ap,
                       const int32_t *__restrict__ Aj, const ValT *__restrict__ Ax,
                       const ValT *__restrict__ x, ValT *__restrict__ y,
                       const ValT *__restrict__ alpha_dev, const ValT *__restrict__ beta_dev,
                       PeerOut peers, const int32_t *__restrict__ coords_x,
                       int32_t *__restrict__ carry_row, ValT *__restrict__ carry_val) {
    constexpr int IPT = kMergeIPT;
    __shared__ __align__(16) ValT s_scan[kSlots];
    __shared__ __align__(16) unsigned char s_flag[kSlots];
    __shared__ ValT s_wval[kMergeBlock / 32];
    __shared__ int s_wflag[kMergeBlock / 32];

    const int tid = threadIdx.x;
    const int64_t tile = blockIdx.x;
    const int64_t total = (int64_t)n_rows + (int64_t)nnz;
    const int64_t d0 = tile * kMergeTile;
    const int64_t d1 = d0 + kMergeTile < total ? d0 + kMergeTile : total;
    const int32_t sx = __ldg(coords_x + tile);
    const int32_t ex = __ldg(coords_x + tile + 1);
    const int64_t sy = d0 - sx;
    const int R = ex - sx;
    const int Z = (int)((d1 - ex) - sy);
    const int shift = (int)(sy & 3);
    const int64_t a0 = sy - shift;
    const ValT ident = S::identity();

    *reinterpret_cast<uint2 *>(s_flag + tid * IPT) = make_uint2(0u, 0u);
    const int slot0 = tid * IPT;
    const uint64_t pol_stream = policy_evict_first();
    const uint64_t pol_x = policy_evict_last();
    int c[IPT];
    ValT p[IPT];
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        c[k] = 0;
        p[k] = (ValT)0;
    }
    if (slot0 < shift + Z) {
        const int64_t g = a0 + slot0;
        if (g + IPT <= (int64_t)nnz) {
            const int4 ca = ldg_stream_int4(Aj + g, pol_stream);
            const int4 cb = ldg_stream_int4(Aj + g + 4, pol_stream);
            c[0] = ca.x; c[1] = ca.y; c[2] = ca.z; c[3] = ca.w;
            c[4] = cb.x; c[5] = cb.y; c[6] = cb.z; c[7] = cb.w;
            LoadVals<ValT>::vec8(Ax + g, pol_stream, p);
        } else {
#pragma unroll
            for (int k = 0; k < IPT; ++k) {
                if (g + k < (int64_t)nnz) {
                    c[k] = __ldg(Aj + g + k);
                    p[k] = __ldg(Ax + g + k);
                }
            }
        }
    }
    const ValT alpha = (S::kLinear && alpha_dev) ? __ldg(alpha_dev) : (ValT)1;
    const ValT beta = (S::kLinear && beta_dev) ? __ldg(beta_dev) : (ValT)0;
    __syncthreads();
    for (int j = tid; j < R; j += kMergeBlock) {
        const int64_t q = (int64_t)__ldg(Ap + sx + 1 + j) - sy;
        if (q < Z) s_flag[(int)q + shift] = 1;
    }
    {
        ValT xv[IPT];
#pragma unroll
        for (int k = 0; k < IPT; ++k) {
            const int i = slot0 + k - shift;
            xv[k] = (i >= 0 && i < Z) ? ldg_hint(x + c[k], pol_x) : (ValT)0;
        }
#pragma unroll
        for (int k = 0; k < IPT; ++k) {
            const int i = slot0 + k - shift;
            p[k] = (i >= 0 && i < Z) ? S::combine(p[k], xv[k]) : ident;
        }
    }
    __syncthreads();

    const uint2 fw = *reinterpret_cast<const uint2 *>(s_flag + slot0);
    const unsigned long long fbits = ((unsigned long long)fw.y << 32) | fw.x;
    int flag = fbits != 0ull;
    ValT val = ident;
#pragma unroll
    for (int k = 0; k < IPT; ++k) val = ((fbits >> (8 * k)) & 1ull) ? p[k] : S::reduce(val, p[k]);
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const ValT pvv = __shfl_up_sync(0xffffffffu, val, d);
        const int pf = __shfl_up_sync(0xffffffffu, flag, d);
        if (lane >= d) {
            if (!flag) val = S::reduce(pvv, val);
            flag |= pf;
        }
    }
    if (lane == 31) {
        s_wval[warp] = val;
        s_wflag[warp] = flag;
    }
    ValT ev = __shfl_up_sync(0xffffffffu, val, 1);
    int ef = __shfl_up_sync(0xffffffffu, flag, 1);
    if (lane == 0) {
        ev = ident;
        ef = 0;
    }
    __syncthreads();
    ValT wv = ident;
#pragma unroll
    for (int w = 0; w < kMergeBlock / 32; ++w) {
        if (w < warp) {
            const ValT v = s_wval[w];
            wv = s_wflag[w] ? v : S::reduce(wv, v);
        }
    }
    ValT run = ef ? ev : S::reduce(wv, ev);
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        run = ((fbits >> (8 * k)) & 1ull) ? p[k] : S::reduce(run, p[k]);
        p[k] = run;
    }
    sts8(s_scan + slot0, p);
    __syncthreads();

    const ValT *scan = s_scan + shift;
    for (int j = tid; j < R; j += kMergeBlock) {
        const int64_t b64 = (int64_t)__ldg(Ap + sx + j) - sy;
        const int q = (int)((int64_t)__ldg(Ap + sx + 1 + j) - sy);
        const int b = b64 > 0 ? (int)b64 : 0;
        const ValT sum = q > b ? scan[q - 1] : ident;
        ValT out = S::kLinear ? alpha * sum : sum;
        if (S::kLinear && beta_dev && beta != (ValT)0) out += beta * y[(int64_t)sx + j];  // beta = 0: y is not read (BLAS)
        // beta makes every row's value depend on the old y, and a non-zero identity makes empty
        // rows non-zero: in both cases every row goes to the peers
        store_y_nonempty(y, peers, (int64_t)sx + j, out, q > b || beta_dev != nullptr || !S::kLinear);
    }
    if (tid == 0) {
        const int64_t lq = R > 0 ? (int64_t)__ldg(Ap + ex) - sy : 0;
        const int lastq = lq > 0 ? (int)lq : 0;
        carry_row[tile] = ex;
        carry_val[tile] = Z > lastq ? scan[Z - 1] : ident;
    }
}

template <typename S, typename ValT>
__global__ void __launch_bounds__(256)
merge_fixup_genl_kernel(int32_t n_rows, int64_t num_tiles, const int32_t *__restrict__ carry_row,
                        const ValT *__restrict__ carry_val, ValT *__restrict__ y,
                        const ValT *__restrict__ alpha_dev, PeerOut peers) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= num_tiles) return;
    const int32_t row = carry_row[t];
    if (row >= n_rows) return;
    if (t > 0 && carry_row[t - 1] == row) return;
    ValT sum = carry_val[t];
    for (int64_t u = t + 1; u < num_tiles && carry_row[u] == row; ++u) sum = S::reduce(sum, carry_val[u]);
    if (S::kLinear) {
        const ValT alpha = alpha_dev ? __ldg(alpha_dev) : (ValT)1;
        store_y(y, peers, (int64_t)row, y[row] + alpha * sum);
    } else {
        store_y(y, peers, (int64_t)row, S::reduce(y[row], sum));
    }
}

}  // namespace

template <typename S, typename OffT, typename ValT>
static int launch_merge_genl_s(const SpmvProblem<OffT, ValT> &p, const ValT *beta_dev) {
    const int64_t total = (int64_t)p.n_rows + (int64_t)p.nnz;
    const int64_t num_tiles = (total + kMergeTile - 1) / kMergeTile;
    if (num_tiles <= 0) return SPMVB200_OK;
    if (num_tiles > 0x7fffffffLL) return SPMVB200_ERR_UNSUPPORTED;
    void *coords = nullptr, *crow = nullptr, *cval = nullptr;
    SPMV_TRY(scratch_get(p.stream, SCRATCH_COORDS, (size_t)(num_tiles + 1) * sizeof(int32_t), &coords));
    SPMV_TRY(scratch_get(p.stream, SCRATCH_CARRY_ROW, (size_t)num_tiles * sizeof(int32_t), &crow));
    SPMV_TRY(scratch_get(p.stream, SCRATCH_CARRY_VAL, (size_t)num_tiles * sizeof(ValT), &cval));
    SPMV_TRY(launch_partition<OffT>(p.n_rows, p.nnz, p.Ap, kMergeTile, num_tiles + 1,
                                    static_cast<int32_t *>(coords), p.stream));
    {
        KernelTimerScope timed(p.stream);
        merge_tile_genl_kernel<S, OffT, ValT><<<(unsigned)num_tiles, kMergeBlock, 0, p.stream>>>(
            p.n_rows, p.nnz, p.Ap, p.Aj, p.Ax, p.x, p.y, p.alpha_dev, beta_dev, p.peers,
            (const int32_t *)coords, static_cast<int32_t *>(crow), static_cast<ValT *>(cval));
    }
    SPMV_LAUNCH_CHECK();
    if (num_tiles > 1) {
        const int64_t blocks = (num_tiles + 255) / 256;
        merge_fixup_genl_kernel<S, ValT><<<(unsigned)blocks, 256, 0, p.stream>>>(
            p.n_rows, num_tiles, (const int32_t *)crow, (const ValT *)cval, p.y, p.alpha_dev, p.peers);
        SPMV_LAUNCH_CHECK();
    }
    return SPMVB200_OK;
}

template <typename OffT, typename ValT>
int launch_merge_genl(const SpmvProblem<OffT, ValT> &p, int semiring, const ValT *beta_dev) {
    if (semiring != SPMVB200_SEMIRING_PLUS_TIMES && (p.alpha_dev || beta_dev)) return SPMVB200_ERR_UNSUPPORTED;
    switch (semiring) {
        case SPMVB200_SEMIRING_PLUS_TIMES: return launch_merge_genl_s<SrPlusTimes<ValT>>(p, beta_dev);
        case SPMVB200_SEMIRING_MIN_PLUS: return launch_merge_genl_s<SrMinPlus<ValT>>(p, beta_dev);
        case SPMVB200_SEMIRING_MAX_PLUS: return launch_merge_genl_s<SrMaxPlus<ValT>>(p, beta_dev);
        case SPMVB200_SEMIRING_OR_AND: return launch_merge_genl_s<SrOrAnd<ValT>>(p, beta_dev);
        default: return SPMVB200_ERR_INVALID;
    }
}
template int launch_merge_genl<int32_t, float>(const SpmvProblem<int32_t, float> &, int, const float *);
template int launch_merge_genl<int32_t, double>(const SpmvProblem<int32_t, double> &, int, const double *);
template int launch_merge_genl<int64_t, float>(const SpmvProblem<int64_t, float> &, int, const float *);
template int launch_merge_genl<int64_t, double>(const SpmvProblem<int64_t, double> &, int, const double *);

template <typename OffT>
int launch_partition(int32_t n_rows, OffT nnz, const OffT *Ap, int64_t tile_items, int64_t n_coords,
                     int32_t *coords_x, cudaStream_t stream, bool reuse) {
    if (n_coords <= 0) return SPMVB200_OK;
    // reuse: the caller vouches that Ap still holds what it held when these coordinates were
    // written (same pointers, same sizes, same stream) -- nothing to search again
    const PartitionTag tag{coords_x, Ap, (int64_t)n_rows, (int64_t)nnz, tile_items, n_coords};
    if (reuse && partition_tag_matches(stream, tag)) return SPMVB200_OK;
    const int64_t blocks = (n_coords + 255) / 256;
    // optionally on a side stream (option "side_stream", off: see side_fork in common.cuh)
    cudaStream_t side = nullptr;
    SPMV_TRY(side_fork(stream, &side));
    merge_partition_kernel<OffT><<<(unsigned)blocks, 256, 0, side>>>(n_rows, nnz, Ap, tile_items,
                                                                     n_coords, coords_x);
    SPMV_LAUNCH_CHECK();
    SPMV_TRY(side_join(stream));
    partition_tag_store(stream, tag);
    return SPMVB200_OK;
}
template int launch_partition<int32_t>(int32_t, int32_t, const int32_t *, int64_t, int64_t,
                                       int32_t *, cudaStream_t, bool);
template int launch_partition<int64_t>(int32_t, int64_t, const int64_t *, int64_t, int64_t,
                                       int32_t *, cudaStream_t, bool);

// CTA size of the register-staged tile kernel: 128 threads (1020-item tiles) -- measured: 128 is
// 3-8 % faster than 256 on c2/c3/c4 (shorter barrier waits, 16 CTAs per SM) and, since the hot-x
// plan, 4 % faster on c5 as well.
// 64-bit offsets used 256-thread CTAs (2044-item tiles) while R-MAT scale 27 was bound by the TLB
// and the DRAM (2 % ahead of 128 there); with the hot-x plan the kernel is L1TEX-bound like the
// 32-bit one and 128 threads win: tile kernel 10.74 -> 10.31 ms, step 10.92 -> 10.52 ms.
#ifndef SPMV_MERGE_O64_BLOCK
#define SPMV_MERGE_O64_BLOCK 128
#endif
template <typename OffT> constexpr int merge_reg_block() { return sizeof(OffT) == 4 ? 128 : SPMV_MERGE_O64_BLOCK; }

int64_t merge_tile_items(int offset_bits) {
    if (option_get("merge_staging", 0) == 1) return kMergeTile;
    return (offset_bits == 32 ? merge_reg_block<int32_t>() : merge_reg_block<int64_t>()) * kMergeIPT - 4;
}

template <typename OffT, typename ValT>
int launch_merge(const SpmvProblem<OffT, ValT> &p) {
    const bool tma = option_get("merge_staging", 0) == 1;
    constexpr int RB = merge_reg_block<OffT>();
    const int tile_items = tma ? kMergeTile : RB * kMergeIPT - 4;
    const int64_t total = (int64_t)p.n_rows + (int64_t)p.nnz;
    const int64_t num_tiles = (total + tile_items - 1) / tile_items;
    if (num_tiles <= 0) return SPMVB200_OK;
    if (num_tiles > 0x7fffffffLL) return SPMVB200_ERR_UNSUPPORTED;

    void *coords = nullptr, *crow = nullptr, *cval = nullptr;
    SPMV_TRY(scratch_get(p.stream, SCRATCH_COORDS, (size_t)(num_tiles + 1) * sizeof(int32_t), &coords));
    SPMV_TRY(scratch_get(p.stream, SCRATCH_CARRY_ROW, (size_t)num_tiles * sizeof(int32_t), &crow));
    SPMV_TRY(scratch_get(p.stream, SCRATCH_CARRY_VAL, (size_t)num_tiles * sizeof(ValT), &cval));

    SPMV_TRY(launch_partition<OffT>(p.n_rows, p.nnz, p.Ap, tile_items, num_tiles + 1,
                                    static_cast<int32_t *>(coords), p.stream, p.reuse_partition));

    // shared-memory carveout in percent of 228 KB; -1 = the driver's choice, -2 (default) = 64 KB
    // for fp32 and the driver's choice for fp64.  The driver picks 100 KB to fit every CTA the
    // registers allow, but the L1 half of the array is what holds the gathers in flight: R-MAT
    // scale 27 15.04 ms at 100 KB, 14.70 at 64 KB, 14.87 at 32 KB, 16.4 at 132 KB; scale 24
    // 1187 / 1146 / 1289 us.  fp64 tiles are twice as large and lose too many CTAs at 64 KB
    // (65536 x 2048 fp64: 728 -> 796 us).
    int64_t carveout = option_get("merge_carveout", -2);
    if (carveout == -2) carveout = sizeof(ValT) == 4 ? 28 : -1;
    LaunchCfg lc;
    // "merge_staging": 0 (default) = Aj/Ax into registers, 1 = TMA bulk copies into shared
    // memory (kept for the ablation that decided against it; see merge_tile_reg_body)
    if (tma) {
        static int64_t attr_carveout = -3;  // per instantiation: last carveout applied
        constexpr size_t smem = merge_smem_bytes<OffT, ValT>();
        if (attr_carveout != carveout) {
            SPMV_CUDA_TRY(cudaFuncSetAttribute(merge_tile_tma_kernel<OffT, ValT>,
                                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            SPMV_CUDA_TRY(cudaFuncSetAttribute(merge_tile_tma_kernel<OffT, ValT>,
                                               cudaFuncAttributePreferredSharedMemoryCarveout,
                                               carveout < 0 ? (int)cudaSharedmemCarveoutDefault : (int)carveout));
            attr_carveout = carveout;
        }
        make_launch_cfg(lc, dim3((unsigned)num_tiles), dim3(kMergeBlock), smem, p.stream, p.x,
                        (size_t)p.n_cols * sizeof(ValT));
        KernelTimerScope timed(p.stream);
        SPMV_CUDA_TRY(cudaLaunchKernelEx(&lc.cfg, merge_tile_tma_kernel<OffT, ValT>, p.n_rows, p.nnz,
                                         p.Ap, p.Aj, p.Ax, p.x, p.y, p.alpha_dev, p.peers,
                                         (const int32_t *)coords, static_cast<int32_t *>(crow),
                                         static_cast<ValT *>(cval)));
    } else {
        const bool has_peers = p.peers.n != 0;
        // tile body: "merge_algo" 0 = row markers, 1 = byte flags, -1 (default) by value type.
        // Measured (L2 flushed): fp32 flags 1121 us / markers 1140 us on R-MAT scale 24 (the marker
        // form costs 8 more registers and 2 KB more shared memory per CTA), fp64 746 / 683 us on the
        // 65536 x 2048 matrix (no second pass over Ap, one barrier less).
        const int64_t algo_opt = option_get("merge_algo", -1);
        const bool flags_form = algo_opt < 0 ? sizeof(ValT) == 4 : algo_opt == 1;
        // 16 CTAs of 128 threads per SM need 32 registers: the bound is only applied where ptxas meets
        // it without spilling (fp32: both forms with 32-bit offsets, the marker form with 64-bit;
        // fp64 needs 48-64 registers either way)
        const bool occ = sizeof(ValT) == 4 && (sizeof(OffT) == 4 || !flags_form);
        // multicast peers (one pointer): its own fp32 flag-form variant, 8 CTAs per SM
        const bool mc_f32 = p.peers.n < 0 && sizeof(ValT) == 4 && flags_form;
        // hot-x plan (hotx.cu): by default only for a caller that vouches for an unchanged matrix.
        // Two uses of it.  (a) x far longer than the TLB and the L2 reach ("hot_x_min_bytes"): up to
        // "hot_x_max_bytes" of the most frequent columns' x in one dense array.  (b) whatever the
        // size of x: the few thousand most frequent columns in a shared-memory table of the
        // persistent tile kernel (merge_tile_table_kernel; "hot_x_table" -1 = fp32 only, 0 = off,
        // 1 = on; "hot_x_table_bytes" = the kernel's dynamic shared memory, tiles and table).
        const int64_t hot_opt = option_get("hot_x", -1);
        const int64_t tbl_opt = option_get("hot_x_table", -1);
        // by default only where the persistent grid has work for every SM: at least four rounds of
        // tiles per group (4.8 M path items on 148 SMs); a smaller matrix is spread over more SMs by
        // one CTA per tile
        const DeviceInfo *tdi = nullptr;
        SPMV_TRY(current_device_info(&tdi));
        const bool tbl_ok = RB == kTableBlock &&
                            (tbl_opt > 0 || (tbl_opt < 0 && sizeof(ValT) == 4 && flags_form &&
                                             num_tiles >= (int64_t)tdi->sm_count * kTableGroups * 4));
        constexpr bool desc_used = tile_desc_used<kTableGroups, OffT, ValT>();
        constexpr int64_t flag_smem = (int64_t)kTableGroups * kTableBlock * kMergeIPT;
        constexpr int64_t tile_smem = (int64_t)sizeof(TileSmem<kTableBlock, ValT>) * kTableGroups +
                                      (desc_used ? 0 : flag_smem);
        // What the option charges per tile in flight: its shared memory and its 1 KB of row-start
        // flags, also where the start mask replaces them, so that the option gives the table sizes
        // measured below either way.  At the defaults the 8 KB left over do not move the carveout off
        // its step (100 KB), so the L1 does not gain them either.
        constexpr int64_t tile_charge = (int64_t)sizeof(TileSmem<kTableBlock, ValT>) * kTableGroups + flag_smem;
        // The option is per SM (every CTA has 1 KB reserved by the system inside a carveout size);
        // -1 = by the size of x.  What the table takes, the L1 loses, in the carveout's steps
        // (100 / 132 / 164 / 196 KB): while x sits in the L2 (R-MAT scale 24) 163 KB is the best size
        // and the next step a cliff (1100 us plain, 1035 / 1011 / 1000 / 1134 us at 99 / 131 / 163 /
        // 179 KB); with x in DRAM (scale 27) the misses in flight need the L1 more than the gathers
        // need the table (11.4 ms plain, 10.3 / 10.4 / 11.0 ms at 83 / 99 / 115 KB).
        const bool big_x = (int64_t)p.n_cols * (int64_t)sizeof(ValT) > option_get("hot_x_min_bytes", 256ll << 20);
        int64_t tbl_bytes = option_get("hot_x_table_bytes", -1);
        if (tbl_bytes < 0) tbl_bytes = big_x ? 99 << 10 : 163 << 10;
        if (tbl_bytes > 226 << 10) tbl_bytes = 226 << 10;
        tbl_bytes = (tbl_bytes + 1024) / kTableCtas - 1024;
        const int64_t k_table = tbl_ok && tbl_bytes > tile_charge ? (tbl_bytes - tile_charge) / (int64_t)sizeof(ValT) : 0;
        const bool want_hot = hot_opt > 0 || (hot_opt < 0 && p.reuse_partition && (big_x || k_table > 0));
        const int64_t k_max = (hot_opt > 0 || big_x) ? option_get("hot_x_max_bytes", 32 << 20) / (int64_t)sizeof(ValT)
                                                     : k_table;
        const HotPlan *hot = nullptr;
        if (want_hot) SPMV_TRY(hot_plan_get(p.Aj, (int64_t)p.nnz, p.n_cols, k_max, k_table, p.stream, true, &hot));
        // a call without the flag says "this may be a new matrix": a plan left at this address by
        // an earlier one must not survive it
        else if (hot_opt < 0 && !p.reuse_partition) hot_plan_drop(p.Aj);
        make_launch_cfg(lc, dim3((unsigned)num_tiles), dim3(RB), 0, p.stream, p.x,
                        (size_t)p.n_cols * sizeof(ValT));
        if (hot) {
            const ValT *x_hot = nullptr;
            SPMV_TRY(hot_gather<ValT>(*hot, p.x, p.stream, &x_hot));
            const ValT *x_hot_biased = x_hot - ((ptrdiff_t)1 << 31);
            if (k_table > 0 && hot->K_table > 0) {
                auto tkernel = p.peers.n < 0 ? merge_tile_table_kernel<2, OffT, ValT>
                               : has_peers   ? merge_tile_table_kernel<1, OffT, ValT>
                                             : merge_tile_table_kernel<0, OffT, ValT>;
                int64_t tn = hot->K_table < k_table ? hot->K_table : k_table;
                const int64_t cap = option_get("hot_x_table_limit", -1);   // experiments: fewer entries than planned
                if (cap >= 0 && cap < tn) tn = cap;
                const uint32_t table_n = (uint32_t)tn;
                // the tile descriptors: built once per search of the partition, reused with it
                void *row_end = nullptr, *start_mask = nullptr;
                constexpr int64_t mask_bytes = kTableBlock * kMergeIPT / 8;
                if (desc_used) {
                    SPMV_TRY(scratch_get(p.stream, SCRATCH_ROW_END, (size_t)p.n_rows * sizeof(uint16_t), &row_end));
                    SPMV_TRY(scratch_get(p.stream, SCRATCH_START_MASK, (size_t)(num_tiles * mask_bytes), &start_mask));
                }
                if (desc_used && !tile_desc_current(p.stream, row_end, start_mask)) {
                    SPMV_CUDA_TRY(cudaMemsetAsync(start_mask, 0, (size_t)(num_tiles * mask_bytes), p.stream));
                    if (p.n_rows > 0) {
                        tile_desc_kernel<OffT><<<(unsigned)(((int64_t)p.n_rows + 255) / 256), 256, 0, p.stream>>>(
                            p.n_rows, p.nnz, p.Ap, (const int32_t *)coords, static_cast<uint16_t *>(row_end),
                            static_cast<uint32_t *>(start_mask));
                        SPMV_LAUNCH_CHECK();
                    }
                    tile_desc_store(p.stream, row_end, start_mask);
                }
                const TileDesc desc{static_cast<const uint16_t *>(row_end),
                                    static_cast<const unsigned char *>(start_mask)};
                const size_t smem = (size_t)tile_smem + (size_t)table_n * sizeof(ValT);
                SPMV_TRY(apply_max_dynamic_smem(reinterpret_cast<const void *>(tkernel), (int64_t)smem));
                const DeviceInfo *di = tdi;
                const int64_t want_ctas = (num_tiles + kTableGroups - 1) / kTableGroups;
                const int64_t max_ctas = (int64_t)di->sm_count * kTableCtas;
                make_launch_cfg(lc, dim3((unsigned)(want_ctas < max_ctas ? want_ctas : max_ctas)),
                                dim3(kTableGroups * kTableBlock), smem, p.stream, p.x, (size_t)p.n_cols * sizeof(ValT));
                KernelTimerScope timed(p.stream);
                SPMV_CUDA_TRY(cudaLaunchKernelEx(&lc.cfg, tkernel, p.n_rows, p.nnz, p.Ap, hot->Aj2, p.Ax, p.x, p.y,
                                                 p.alpha_dev, p.peers, (const int32_t *)coords,
                                                 static_cast<int32_t *>(crow), static_cast<ValT *>(cval),
                                                 x_hot_biased, x_hot, table_n, num_tiles, desc));
            } else {
            auto kernel = flags_form ? (mc_f32    ? merge_tile_hot_kernel<1, RB, 2, OffT, ValT>
                                        : has_peers ? merge_tile_hot_kernel<1, RB, 1, OffT, ValT>
                                                  : merge_tile_hot_kernel<1, RB, 0, OffT, ValT>)
                                     : (has_peers ? merge_tile_hot_kernel<0, RB, 1, OffT, ValT>
                                        : occ     ? merge_tile_hot_kernel_occ8<0, RB, 0, OffT, ValT>
                                                  : merge_tile_hot_kernel<0, RB, 0, OffT, ValT>);
            SPMV_TRY(apply_carveout(reinterpret_cast<const void *>(kernel), carveout));
            KernelTimerScope timed(p.stream);
            SPMV_CUDA_TRY(cudaLaunchKernelEx(&lc.cfg, kernel, p.n_rows, p.nnz, p.Ap, hot->Aj2, p.Ax, p.x, p.y,
                                             p.alpha_dev, p.peers, (const int32_t *)coords,
                                             static_cast<int32_t *>(crow), static_cast<ValT *>(cval),
                                             x_hot_biased));
            }
        } else {
            auto kernel = flags_form ? (mc_f32    ? merge_tile_reg_kernel<1, RB, 2, OffT, ValT>
                                        : has_peers ? merge_tile_reg_kernel<1, RB, 1, OffT, ValT>   // 40 regs, no spill
                                        : occ     ? merge_tile_reg_kernel_occ8<1, RB, 0, OffT, ValT>
                                                  : merge_tile_reg_kernel<1, RB, 0, OffT, ValT>)
                                     : (has_peers ? merge_tile_reg_kernel<0, RB, 1, OffT, ValT>
                                        : occ     ? merge_tile_reg_kernel_occ8<0, RB, 0, OffT, ValT>
                                                  : merge_tile_reg_kernel<0, RB, 0, OffT, ValT>);
            SPMV_TRY(apply_carveout(reinterpret_cast<const void *>(kernel), carveout));
            KernelTimerScope timed(p.stream);
            SPMV_CUDA_TRY(cudaLaunchKernelEx(&lc.cfg, kernel, p.n_rows, p.nnz, p.Ap, p.Aj, p.Ax, p.x, p.y,
                                             p.alpha_dev, p.peers, (const int32_t *)coords,
                                             static_cast<int32_t *>(crow), static_cast<ValT *>(cval)));
        }
    }
    SPMV_LAUNCH_CHECK();

    if (num_tiles > 1) {
        const int64_t blocks = (num_tiles + 255) / 256;
        merge_fixup_kernel<ValT><<<(unsigned)blocks, 256, 0, p.stream>>>(
            p.n_rows, num_tiles, (const int32_t *)crow, (const ValT *)cval, p.y, p.alpha_dev, p.peers);
        SPMV_LAUNCH_CHECK();
    }
    return SPMVB200_OK;
}

template int launch_merge<int32_t, float>(const SpmvProblem<int32_t, float> &);
template int launch_merge<int32_t, double>(const SpmvProblem<int32_t, double> &);
template int launch_merge<int64_t, float>(const SpmvProblem<int64_t, float> &);
template int launch_merge<int64_t, double>(const SpmvProblem<int64_t, double> &);

}  // namespace spmvb200
