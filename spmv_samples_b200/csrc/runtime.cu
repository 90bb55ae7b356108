// runtime.cu -- host-side runtime of libspmvb200: error slots, device properties, the
// per-(device, stream) scratch cache, tunables, launch counter, launch attributes.
//
// Replaces the reference's per-call cudaMalloc/cudaFree of temporaries
// (reference/include/spmv/cusparse.cuh:72,88; cub_merge.cuh:43,54; LightSpMV.cuh:274,314;
// merge_based/merge_based.cuh:34,46 -- the last one leaks) with buffers that are allocated
// once and grown on demand, so the steady-state call makes no allocation and no sync.
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "common.cuh"

namespace spmvb200 {

namespace {
std::mutex g_mu;
thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};
std::map<int, DeviceInfo> g_devs;

struct ScratchBuf {
    void *ptr = nullptr;
    size_t bytes = 0;
};
struct ScratchSet {
    ScratchBuf slot[SCRATCH_NUM_SLOTS];
    PartitionTag last_partition{nullptr, nullptr, -1, -1, -1, -1};
    const void *tile_desc[2] = {nullptr, nullptr};  // where the descriptors of last_partition are
};
std::map<std::pair<int, cudaStream_t>, ScratchSet> g_scratch;

std::map<std::string, int64_t> &options() {
    static std::map<std::string, int64_t> o = {
        {"l2_window", 0},        // 1: attach an L2 access-policy persistence window over x
        {"vector_width", 0},     // 0: from row statistics; else force lanes per row (1..32)
        {"vector_rows_per_subwarp", 0},  // 0/1: one row per sub-warp; 4: interleaved ablation kernel
        {"light_width", 0},      // same for the dynamic-row kernel
        {"light_rows_per_claim", 0},  // 0: automatic
        {"time_main_kernel", 0}, // 1: cudaEvent bracket around each call's dominant kernel
        {"merge_carveout", -2},  // shared-memory carveout (percent) of the merge tile kernel; -1: driver's, -2: by type
        {"l2_fetch_granularity", 0},  // 32/64/128: cudaLimitMaxL2FetchGranularity; 0 = leave
        {"spmm_force_vector", 0},     // 1: SpMM always takes the row-per-sub-warp kernel
        {"spmm_by_columns", 0},       // 1: merge-class SpMM as K merge-path SpMVs (ablation)
        {"spmm_force_merge", 0},      // 1: SpMM always takes the merge-path tile kernel
        {"spmm_carveout", -1},        // shared-memory carveout (percent) of the merge-path SpMM kernel
        {"merge_staging", 0},    // 0: Aj/Ax into registers (default); 1: TMA bulk copies to smem
        {"auto_kind", -1},       // -1: selector decides; else force a SPMVB200_KIND_*
        {"cusparse_preprocess", 0},  // 1: run cusparseSpMV_preprocess when a plan is built.  Only
                                     // safe while the matrix contents behind (Ap, Aj, Ax) do not
                                     // change; bench.py turns it on for the baseline timing
        {"merge_algo", -1},      // tile body of the merge-path kernel: 0 = row markers, 1 = byte flags, -1 = by value type
        {"hot_x", -1},           // compacted hot part of x in the merge-path kernel: -1 = when the caller
                                 // passes SPMVB200_FLAG_STATIC_PATTERN and x is longer than
                                 // "hot_x_min_bytes"; 0 = never; 1 = always (plan keyed on the Aj pointer)
        {"hot_x_min_bytes", 256ll << 20},
        {"hot_x_table", -1},     // shared-memory table of the most frequent columns (persistent merge tile kernel):
                                 // -1 = fp32 flag form, 0 = never, 1 = always
        {"hot_x_table_limit", -1},  // experiments: use at most this many table entries (0: persistent kernel, no table)
        {"hot_x_table_bytes", -1},  // dynamic shared memory of that kernel (8 tiles in flight + table); -1 = by the size of x
        {"assume_static_pattern", 0},  // 1: every call is treated as carrying SPMVB200_FLAG_STATIC_PATTERN
        {"side_stream", 0},      // 1: small kernels a big one depends on (partition, x_hot refill) run on a side
                                 // stream forked / joined with events (measured: no gain outside the profiler)
        {"hot_x_fill", 0},       // how x_hot is refilled: 0/1 = gather x[hot_cols[r]], 2 = sweep over x, 3 = not at all (experiments)
        {"hot_x_max_bytes", 32ll << 20},   // size of the dense copy of the hot columns' x
        {"power_exchange", -1},    // spmvb200_power_*: 0 = peer stores, 1 = NVLink multicast, -1 = multicast where available
        {"stream_ctas_per_sm", 3},  // persistent CTAs per SM of the CSR-stream kernel
        {"cusparse_alg", 0},     // 0: CUSPARSE_SPMV_ALG_DEFAULT (the reference's call), 1: CSR_ALG1, 2: CSR_ALG2
    };
    // SPMVB200_OPTS="name=value,name=value": presets for callers without an option API of their
    // own (the C++ driver), read once
    static bool env_read = false;
    if (!env_read) {
        env_read = true;
        if (const char *e = std::getenv("SPMVB200_OPTS")) {
            std::string s(e);
            size_t pos = 0;
            while (pos < s.size()) {
                size_t end = s.find(',', pos);
                if (end == std::string::npos) end = s.size();
                const std::string kv = s.substr(pos, end - pos);
                const size_t eq = kv.find('=');
                if (eq != std::string::npos) {
                    auto it = o.find(kv.substr(0, eq));
                    if (it != o.end()) it->second = std::atoll(kv.c_str() + eq + 1);
                }
                pos = end + 1;
            }
        }
    }
    return o;
}
}  // namespace

void record_cuda_error(cudaError_t e, const char *what, const char *file, int line) {
    std::snprintf(g_err, sizeof(g_err), "%s:%d: %s -> %s (%s)", file, line, what,
                  cudaGetErrorName(e), cudaGetErrorString(e));
    (void)cudaGetLastError();  // clear the sticky-less error so the next call starts clean
}

const char *last_error() { return g_err; }

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
int64_t launch_count() { return g_launches.load(std::memory_order_relaxed); }

int current_device_info(const DeviceInfo **out) {
    int dev = -1;
    SPMV_CUDA_TRY(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = g_devs.find(dev);
    if (it == g_devs.end()) {
        cudaDeviceProp prop;
        SPMV_CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
        DeviceInfo di;
        di.device = dev;
        di.sm_count = prop.multiProcessorCount;
        di.max_threads_per_sm = prop.maxThreadsPerMultiProcessor;
        di.l2_bytes = (size_t)prop.l2CacheSize;
        di.persisting_l2_max = (size_t)prop.persistingL2CacheMaxSize;
        di.access_window_max = (size_t)prop.accessPolicyMaxWindowSize;
        di.smem_optin = (size_t)prop.sharedMemPerBlockOptin;
        it = g_devs.emplace(dev, di).first;
    }
    *out = &it->second;
    return SPMVB200_OK;
}

int scratch_get(cudaStream_t stream, ScratchSlot slot, size_t bytes, void **out) {
    int dev = -1;
    SPMV_CUDA_TRY(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_mu);
    ScratchBuf &b = g_scratch[{dev, stream}].slot[slot];
    if (bytes < 256) bytes = 256;
    if (b.bytes < bytes) {
        // grow geometrically; the old buffer may still be in use by queued kernels on this
        // stream, so free it stream-ordered
        size_t want = bytes + bytes / 4;
        void *np = nullptr;
        SPMV_CUDA_TRY(cudaMalloc(&np, want));
        // new scratch starts zeroed (the block counter of the norm exchange relies on it)
        SPMV_CUDA_TRY(cudaMemsetAsync(np, 0, want, stream));
        if (b.ptr) {
            SPMV_CUDA_TRY(cudaStreamSynchronize(stream));
            SPMV_CUDA_TRY(cudaFree(b.ptr));
        }
        b.ptr = np;
        b.bytes = want;
    }
    *out = b.ptr;
    return SPMVB200_OK;
}

bool partition_tag_matches(cudaStream_t stream, const PartitionTag &tag) {
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return false;
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = g_scratch.find({dev, stream});
    return it != g_scratch.end() && it->second.last_partition == tag;
}
void partition_tag_store(cudaStream_t stream, const PartitionTag &tag) {
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return;
    std::lock_guard<std::mutex> lk(g_mu);
    ScratchSet &set = g_scratch[{dev, stream}];
    set.last_partition = tag;
    set.tile_desc[0] = set.tile_desc[1] = nullptr;  // new coordinates: the descriptors are stale
}
bool tile_desc_current(cudaStream_t stream, const void *row_end, const void *start_mask) {
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return false;
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = g_scratch.find({dev, stream});
    return it != g_scratch.end() && it->second.tile_desc[0] == row_end && it->second.tile_desc[1] == start_mask;
}
void tile_desc_store(cudaStream_t stream, const void *row_end, const void *start_mask) {
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return;
    std::lock_guard<std::mutex> lk(g_mu);
    ScratchSet &set = g_scratch[{dev, stream}];
    set.tile_desc[0] = row_end;
    set.tile_desc[1] = start_mask;
}

void scratch_release_all() {
    std::lock_guard<std::mutex> lk(g_mu);
    int cur = -1;
    cudaGetDevice(&cur);
    for (auto &kv : g_scratch) {
        cudaSetDevice(kv.first.first);
        cudaDeviceSynchronize();
        for (auto &b : kv.second.slot)
            if (b.ptr) cudaFree(b.ptr);
    }
    g_scratch.clear();
    if (cur >= 0) cudaSetDevice(cur);
}

namespace {
struct SideLane {
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};
// one side stream per (device, caller stream)
std::map<std::pair<int, cudaStream_t>, SideLane> g_lanes;

int side_lane(cudaStream_t stream, SideLane *out) {
    int dev = -1;
    SPMV_CUDA_TRY(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_mu);
    SideLane &l = g_lanes[{dev, stream}];
    if (!l.stream) {
        SPMV_CUDA_TRY(cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking));
        SPMV_CUDA_TRY(cudaEventCreateWithFlags(&l.fork, cudaEventDisableTiming));
        SPMV_CUDA_TRY(cudaEventCreateWithFlags(&l.join, cudaEventDisableTiming));
    }
    *out = l;
    return SPMVB200_OK;
}
}  // namespace

int side_fork(cudaStream_t stream, cudaStream_t *side) {
    if (option_get("side_stream", 0) <= 0) {   // the default: everything on the caller's stream
        *side = stream;
        return SPMVB200_OK;
    }
    SideLane lane;
    SPMV_TRY(side_lane(stream, &lane));
    SPMV_CUDA_TRY(cudaEventRecord(lane.fork, stream));
    SPMV_CUDA_TRY(cudaStreamWaitEvent(lane.stream, lane.fork, 0));
    *side = lane.stream;
    return SPMVB200_OK;
}

int side_join(cudaStream_t stream) {
    if (option_get("side_stream", 0) <= 0) return SPMVB200_OK;
    SideLane lane;
    SPMV_TRY(side_lane(stream, &lane));
    SPMV_CUDA_TRY(cudaEventRecord(lane.join, lane.stream));
    SPMV_CUDA_TRY(cudaStreamWaitEvent(stream, lane.join, 0));
    return SPMVB200_OK;
}

int64_t option_get(const char *name, int64_t fallback) {
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = options().find(name);
    return it == options().end() ? fallback : it->second;
}
int option_set(const char *name, int64_t v) {
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = options().find(name);
    if (it == options().end()) return SPMVB200_ERR_INVALID;
    it->second = v;
    // device-wide limit, applied to the current device when the option is set: a random 4-byte
    // gather that misses L2 only needs one 32-byte sector from HBM, not the default 64 bytes
    if (std::string(name) == "l2_fetch_granularity" && (v == 32 || v == 64 || v == 128))
        cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)v);
    return SPMVB200_OK;
}

// ---- cudaEvent bracket around the dominant kernel (option "time_main_kernel") -----------
namespace {
struct EventPair {
    cudaEvent_t a, b;
};
std::vector<EventPair> g_ev_free, g_ev_pending;
double g_ev_ms = 0.0;
int64_t g_ev_count = 0;

void fold_pending_locked() {
    for (auto &p : g_ev_pending) {
        float ms = 0.f;
        if (cudaEventSynchronize(p.b) == cudaSuccess && cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
            g_ev_ms += ms;
            ++g_ev_count;
        }
        g_ev_free.push_back(p);
    }
    g_ev_pending.clear();
}
}  // namespace

int apply_carveout(const void *kernel, int64_t percent) {
    const DeviceInfo *di = nullptr;
    SPMV_TRY(current_device_info(&di));
    static std::map<std::pair<int, const void *>, int64_t> applied;
    std::lock_guard<std::mutex> lk(g_mu);
    auto key = std::make_pair(di->device, kernel);
    auto it = applied.find(key);
    if (it != applied.end() && it->second == percent) return SPMVB200_OK;
    SPMV_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       percent < 0 ? (int)cudaSharedmemCarveoutDefault : (int)percent));
    applied[key] = percent;
    return SPMVB200_OK;
}

int apply_max_dynamic_smem(const void *kernel, int64_t bytes) {
    const DeviceInfo *di = nullptr;
    SPMV_TRY(current_device_info(&di));
    static std::map<std::pair<int, const void *>, int64_t> applied;
    std::lock_guard<std::mutex> lk(g_mu);
    auto key = std::make_pair(di->device, kernel);
    auto it = applied.find(key);
    if (it != applied.end() && it->second >= bytes) return SPMVB200_OK;
    SPMV_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    applied[key] = bytes;
    return SPMVB200_OK;
}

KernelTimerScope::KernelTimerScope(cudaStream_t s) : stream_(s) {
    if (option_get("time_main_kernel", 0) <= 0) return;
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_ev_pending.size() >= 2048) fold_pending_locked();
    EventPair p;
    if (!g_ev_free.empty()) {
        p = g_ev_free.back();
        g_ev_free.pop_back();
    } else if (cudaEventCreate(&p.a) != cudaSuccess || cudaEventCreate(&p.b) != cudaSuccess) {
        return;
    }
    a_ = p.a;
    b_ = p.b;
    active_ = true;
    cudaEventRecord(a_, stream_);
}
KernelTimerScope::~KernelTimerScope() {
    if (!active_) return;
    cudaEventRecord(b_, stream_);
    std::lock_guard<std::mutex> lk(g_mu);
    g_ev_pending.push_back(EventPair{a_, b_});
}
void kernel_timer_read(double *total_ms, int64_t *launches) {
    std::lock_guard<std::mutex> lk(g_mu);
    fold_pending_locked();
    *total_ms = g_ev_ms;
    *launches = g_ev_count;
    g_ev_ms = 0.0;
    g_ev_count = 0;
}

void make_launch_cfg(LaunchCfg &lc, dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                     const void *x, size_t x_bytes) {
    std::memset(&lc, 0, sizeof(lc));
    lc.cfg.gridDim = grid;
    lc.cfg.blockDim = block;
    lc.cfg.dynamicSmemBytes = smem;
    lc.cfg.stream = stream;
    lc.cfg.attrs = lc.attrs;
    lc.cfg.numAttrs = 0;
    if (x && x_bytes && option_get("l2_window", 0) > 0) {
        const DeviceInfo *di = nullptr;
        if (current_device_info(&di) == SPMVB200_OK && di->access_window_max > 0 &&
            di->persisting_l2_max > 0) {
            static std::map<int, bool> limit_set;
            {
                std::lock_guard<std::mutex> lk(g_mu);
                if (!limit_set[di->device]) {
                    cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, di->persisting_l2_max);
                    limit_set[di->device] = true;
                }
            }
            size_t win = x_bytes < di->access_window_max ? x_bytes : di->access_window_max;
            float ratio = win <= di->persisting_l2_max
                              ? 1.0f
                              : (float)((double)di->persisting_l2_max / (double)win);
            cudaLaunchAttribute &a = lc.attrs[lc.cfg.numAttrs++];
            a.id = cudaLaunchAttributeAccessPolicyWindow;
            a.val.accessPolicyWindow.base_ptr = const_cast<void *>(x);
            a.val.accessPolicyWindow.num_bytes = win;
            a.val.accessPolicyWindow.hitRatio = ratio;
            a.val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
            a.val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        }
    }
}

}  // namespace spmvb200

// ------------------------------------------------------------------------ C ABI (misc)
namespace spmvb200 {
const char *last_error();
int64_t launch_count();
int option_set(const char *name, int64_t v);
}  // namespace spmvb200

extern "C" {

const char *spmvb200_status_string(int status) {
    switch (status) {
        case SPMVB200_OK: return "ok";
        case SPMVB200_ERR_INVALID: return "invalid argument";
        case SPMVB200_ERR_ALIGNMENT: return "Ap/Aj/Ax must be 16-byte aligned";
        case SPMVB200_ERR_CUDA: return "CUDA runtime error";
        case SPMVB200_ERR_UNSUPPORTED: return "unsupported configuration";
        case SPMVB200_ERR_CUSPARSE: return "cuSPARSE error";
        default: return "unknown status";
    }
}
const char *spmvb200_last_cuda_error(void) { return spmvb200::last_error(); }
const char *spmvb200_version(void) { return "spmvb200 0.1 (sm_100a)"; }
int spmvb200_set_option(const char *name, int64_t value) { return spmvb200::option_set(name, value); }
int64_t spmvb200_get_option(const char *name) { return spmvb200::option_get(name, -1); }
int64_t spmvb200_launch_count(void) { return spmvb200::launch_count(); }

}  // extern "C"
