// Host-side plumbing shared by the C-ABI entry points and the kernel launchers:
// context (= the caller's OpRunContext + BufferPool), error strings, caching allocator.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <array>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "../../include/rten_b200.h"

struct rten_ctx;
struct rten_graph {
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    uint64_t kernels = 0;  // kernels captured (added to the launch counter on every replay)
    // Pool buffers whose raw pointers are baked into the instantiated graph (temporaries and intermediate outputs
    // allocated or released while capturing).  They stay out of the context's pool until the graph is destroyed:
    // a later allocation can never alias memory that a replay reads or writes.
    rten_ctx* ctx = nullptr;  // null once the owning context is gone
    std::vector<std::pair<void*, size_t>> held;
};

// Device-side caching allocator, stream-ordered on the context stream
// (plays src/buffer_pool.rs: size-bucketed reuse within and across runs).
struct DevicePool {
    std::unordered_map<void*, size_t> live;             // ptr -> bucket size
    std::map<size_t, std::vector<void*>> free_buckets;  // bucket size -> free buffers
    size_t bytes_reserved = 0;
    // Graph capture: buffers released while capturing are recycled only INSIDE that capture (stream order inside the
    // graph keeps that safe) and are handed to the rten_graph at graph_end; buffers handed out while capturing that are
    // still live at graph_end are pinned to the graph and join its `held` list when the caller frees them.
    std::map<size_t, std::vector<void*>> cap_free;
    std::unordered_map<void*, size_t> cap_touched;      // every buffer handed out or released during the capture
    std::unordered_map<void*, rten_graph*> pinned;      // live buffer -> graph whose nodes reference it

    static size_t bucket(size_t bytes) {
        if (bytes < 512) bytes = 512;
        if (bytes <= (1u << 20)) {
            size_t b = 512;
            while (b < bytes) b <<= 1;
            return b;
        }
        const size_t mb = 1u << 20;
        return (bytes + mb - 1) / mb * mb;
    }
};

struct rten_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int num_sms = 148;
    int f32_mode = RTEN_F32_TF32X3;  // fp32-grade by default; single-pass TF32 is an explicit opt-in
    uint64_t launches = 0;
    bool capturing = false;
    uint64_t capture_start_launches = 0;
    std::string err;
    DevicePool pool;
    // scratch released at the end of each op call
    std::vector<void*> temps;
    void* trace = nullptr;         // device buffer of 4 x 2048 int64 timestamps (debug), or null
    void* encode_tiled = nullptr;  // cuTensorMapEncodeTiled (driver entry point)
    void* sk_counters = nullptr;   // split-K arrival counters (zero between launches)
    bool autotune = false;         // time candidate launch plans on first sight of a problem (umma_gemm.cu)
    std::map<std::vector<long long>, std::array<int, 8>> tune_cache;
    size_t tune_loaded = 0;        // entries read from RTEN_B200_TUNE_FILE (the file is rewritten when more exist at destroy)
    std::vector<rten_graph*> graphs;  // graphs captured on this context that still exist
    void* attn_cnt = nullptr;      // arrival counters of the split single-query attention kernel (zero between launches)
    int attn_cnt_len = 0;
    uint64_t forced_hits = 0, forced_misses = 0;  // RTEN_B200_FORCE_* launches that found / did not find a matching plan
};

namespace rtb {

// ---- errors -------------------------------------------------------------------------------
inline rten_status fail(rten_ctx* ctx, rten_status st, const char* msg) {
    if (ctx) ctx->err = msg ? msg : "";
    return st;
}
inline rten_status fail_cuda(rten_ctx* ctx, cudaError_t e, const char* where) {
    if (ctx) {
        ctx->err = std::string("CUDA error at ") + where + ": " + cudaGetErrorString(e);
    }
    return RTEN_ERR_CUDA;
}
#define RTB_CUDA(ctx, expr)                                         \
    do {                                                            \
        cudaError_t _e = (expr);                                    \
        if (_e != cudaSuccess) return rtb::fail_cuda(ctx, _e, #expr); \
    } while (0)
#define RTB_TRY(expr)                      \
    do {                                   \
        rten_status _s = (expr);           \
        if (_s != RTEN_OK) return _s;      \
    } while (0)

// ---- allocator ----------------------------------------------------------------------------
rten_status pool_alloc(rten_ctx* ctx, size_t bytes, void** out);
rten_status pool_free(rten_ctx* ctx, void* p);
// temp = freed automatically by release_temps() at the end of the op
rten_status temp_alloc(rten_ctx* ctx, size_t bytes, void** out);
void release_temps(rten_ctx* ctx);

// ---- tensor helpers -----------------------------------------------------------------------
inline int dtype_size(int dt) { return (dt == RTEN_F32 || dt == RTEN_I32) ? 4 : 1; }
inline int64_t numel(const rten_tensor* t) {
    int64_t n = 1;
    for (int i = 0; i < t->ndim; i++) n *= t->shape[i];
    return n;
}
inline bool is_contiguous(const rten_tensor* t) {
    int64_t s = 1;
    for (int i = t->ndim - 1; i >= 0; i--) {
        if (t->shape[i] != 1 && t->strides[i] != s) return false;
        s *= t->shape[i];
    }
    return true;
}
inline void set_contiguous(rten_tensor* t) {
    int64_t s = 1;
    for (int i = t->ndim - 1; i >= 0; i--) {
        t->strides[i] = s;
        s *= t->shape[i];
    }
}
// number of elements spanned from data (positive strides)
inline int64_t span_elems(const rten_tensor* t) {
    if (numel(t) == 0) return 0;
    int64_t s = 1;
    for (int i = 0; i < t->ndim; i++) s += (t->shape[i] - 1) * t->strides[i];
    return s;
}

inline void count_launch(rten_ctx* ctx, int n = 1) { ctx->launches += (uint64_t)n; }

// cross-rank min / max of the DynamicQuantizeLinear range (comm.cu)
rten_status comm_allreduce_minmax(rten_ctx* ctx, struct ::rten_comm* comm, int* mm);
struct RangeExchange;
bool comm_range_exchange(struct ::rten_comm* comm, RangeExchange* out);  // true: the quantise kernel exchanges the range itself

// Launch attributes of a cudaLaunchKernelEx launch: programmatic dependent launch (unless RTEN_B200_NO_PDL is set, read
// at every launch) and, with `cluster2`, a 2x1x1 cluster.  `attr` must hold two entries when `cluster2` is set.
inline void fill_launch_attrs(cudaLaunchConfig_t& cfg, cudaLaunchAttribute* attr, bool cluster2) {
    int nattr = 0;
    if (!getenv("RTEN_B200_NO_PDL")) {
        attr[nattr].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[nattr].val.programmaticStreamSerializationAllowed = 1;
        nattr++;
    }
    if (cluster2) {
        attr[nattr].id = cudaLaunchAttributeClusterDimension;
        attr[nattr].val.clusterDim.x = 2;
        attr[nattr].val.clusterDim.y = 1;
        attr[nattr].val.clusterDim.z = 1;
        nattr++;
    }
    cfg.attrs = attr;
    cfg.numAttrs = nattr;
}

}  // namespace rtb
