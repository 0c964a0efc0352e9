// Context, allocator, staging and copy entry points of the C ABI (include/rten_b200.h).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <iterator>

#include "api_util.h"
#include "rowops.h"

namespace rtb {

rten_status pool_alloc(rten_ctx* ctx, size_t bytes, void** out) {
    const size_t b = DevicePool::bucket(bytes);
    if (ctx->capturing) {  // buffers released earlier in this capture first (they stay private to the graph)
        auto ci = ctx->pool.cap_free.find(b);
        if (ci != ctx->pool.cap_free.end() && !ci->second.empty()) {
            *out = ci->second.back();
            ci->second.pop_back();
            ctx->pool.live[*out] = b;
            return RTEN_OK;
        }
    }
    auto it = ctx->pool.free_buckets.find(b);
    if (it != ctx->pool.free_buckets.end() && !it->second.empty()) {
        *out = it->second.back();
        it->second.pop_back();
        ctx->pool.live[*out] = b;
        if (ctx->capturing) ctx->pool.cap_touched[*out] = b;
        return RTEN_OK;
    }
    // During graph capture (relaxed mode) growing the pool is still legal: cudaMalloc is not a stream operation.
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, b);
    if (e != cudaSuccess) return fail_cuda(ctx, e, "cudaMalloc");
    ctx->pool.bytes_reserved += b;
    ctx->pool.live[p] = b;
    if (ctx->capturing) ctx->pool.cap_touched[p] = b;
    *out = p;
    return RTEN_OK;
}

rten_status pool_free(rten_ctx* ctx, void* p) {
    if (!p) return RTEN_OK;
    auto it = ctx->pool.live.find(p);
    if (it == ctx->pool.live.end()) return fail(ctx, RTEN_ERR_INVALID_VALUE, "pointer was not allocated by this context");
    const size_t b = it->second;
    ctx->pool.live.erase(it);
    if (ctx->capturing) {
        // the captured nodes keep this pointer: reusable by later nodes of the SAME capture only
        ctx->pool.cap_touched[p] = b;
        ctx->pool.cap_free[b].push_back(p);
        return RTEN_OK;
    }
    auto pin = ctx->pool.pinned.find(p);
    if (pin != ctx->pool.pinned.end()) {  // referenced by an instantiated graph: parked there until it is destroyed
        pin->second->held.emplace_back(p, b);
        ctx->pool.pinned.erase(pin);
        return RTEN_OK;
    }
    ctx->pool.free_buckets[b].push_back(p);
    return RTEN_OK;
}

// End of a capture: buffers released during it go to the graph (or back to the pool when the capture failed), buffers
// handed out during it that the caller still holds are pinned to the graph.
static void capture_settle(rten_ctx* ctx, rten_graph* g) {
    DevicePool& pool = ctx->pool;
    for (auto& kv : pool.cap_free)
        for (void* p : kv.second) {
            if (g)
                g->held.emplace_back(p, kv.first);
            else
                pool.free_buckets[kv.first].push_back(p);
        }
    if (g)
        for (auto& kv : pool.cap_touched)
            if (pool.live.count(kv.first)) pool.pinned[kv.first] = g;
    pool.cap_free.clear();
    pool.cap_touched.clear();
}

rten_status temp_alloc(rten_ctx* ctx, size_t bytes, void** out) {
    RTB_TRY(pool_alloc(ctx, bytes, out));
    ctx->temps.push_back(*out);
    return RTEN_OK;
}

void release_temps(rten_ctx* ctx) {
    for (void* p : ctx->temps) pool_free(ctx, p);
    ctx->temps.clear();
}

// ---- staging ------------------------------------------------------------------------------
rten_status OpScope::in(const rten_tensor* t, rten_tensor* view) {
    *view = *t;
    if (t->ndim < 0 || t->ndim > RTEN_MAX_DIMS) return fail(ctx, RTEN_ERR_INVALID_VALUE, "tensor rank out of range");
    for (int i = 0; i < t->ndim; i++)
        if (t->shape[i] < 0 || t->strides[i] < 0) return fail(ctx, RTEN_ERR_INVALID_VALUE, "negative shape or stride");
    if (t->device >= 0) {
        if (t->device != ctx->device) return fail(ctx, RTEN_ERR_CUDA, "tensor lives on a different device than the context");
        return RTEN_OK;
    }
    host_involved = true;
    const int64_t span = span_elems(t);
    const size_t bytes = (size_t)span * dtype_size(t->dtype);
    void* d = nullptr;
    RTB_TRY(temp_alloc(ctx, bytes ? bytes : 16, &d));
    if (bytes) RTB_CUDA(ctx, cudaMemcpyAsync(d, t->data, bytes, cudaMemcpyHostToDevice, ctx->stream));
    view->data = d;
    view->device = ctx->device;
    return RTEN_OK;
}

rten_status OpScope::out(rten_tensor* o, int dtype, int ndim, const int64_t* shape, rten_tensor* view,
                         const int64_t* preferred_strides) {
    if (o->data == nullptr) {
        o->dtype = dtype;
        o->ndim = ndim;
        int64_t n = 1;
        for (int i = 0; i < ndim; i++) {
            o->shape[i] = shape[i];
            n *= shape[i];
        }
        if (preferred_strides)
            for (int i = 0; i < ndim; i++) o->strides[i] = preferred_strides[i];
        else
            set_contiguous(o);
        void* d = nullptr;
        RTB_TRY(pool_alloc(ctx, (size_t)(n ? n : 1) * dtype_size(dtype), &d));
        o->data = d;
        o->device = ctx->device;
        *view = *o;
        allocated.push_back(o);
        return RTEN_OK;
    }
    if (o->dtype != dtype) return fail(ctx, RTEN_ERR_UNSUPPORTED_OUTPUT, "output tensor has the wrong element type");
    if (o->ndim != ndim) return fail(ctx, RTEN_ERR_UNSUPPORTED_OUTPUT, "output tensor has the wrong shape");
    for (int i = 0; i < ndim; i++)
        if (o->shape[i] != shape[i]) return fail(ctx, RTEN_ERR_UNSUPPORTED_OUTPUT, "output tensor has the wrong shape");
    if (o->device >= 0) {
        if (o->device != ctx->device) return fail(ctx, RTEN_ERR_CUDA, "tensor lives on a different device than the context");
        *view = *o;
        return RTEN_OK;
    }
    // host output: compute into a contiguous device temp, copy back in finish()
    if (!is_contiguous(o)) return fail(ctx, RTEN_ERR_UNSUPPORTED_OUTPUT, "host output tensors must be contiguous");
    host_involved = true;
    *view = *o;
    set_contiguous(view);
    void* d = nullptr;
    const size_t bytes = (size_t)numel(o) * dtype_size(dtype);
    RTB_TRY(temp_alloc(ctx, bytes ? bytes : 16, &d));
    view->data = d;
    view->device = ctx->device;
    copybacks.push_back({o->data, d, bytes});
    return RTEN_OK;
}

rten_status OpScope::contiguous(const rten_tensor* v, rten_tensor* c) {
    if (is_contiguous(v)) {
        *c = *v;
        return RTEN_OK;
    }
    *c = *v;
    set_contiguous(c);
    void* d = nullptr;
    const int es = dtype_size(v->dtype);
    RTB_TRY(temp_alloc(ctx, (size_t)(numel(v) ? numel(v) : 1) * es, &d));
    c->data = d;
    long long shape[RTEN_MAX_DIMS], ss[RTEN_MAX_DIMS], ds[RTEN_MAX_DIMS];
    for (int i = 0; i < v->ndim; i++) {
        shape[i] = v->shape[i];
        ss[i] = v->strides[i];
        ds[i] = c->strides[i];
    }
    return launch_nd_copy(ctx, es, v->data, d, v->ndim, shape, ss, ds);
}

rten_status OpScope::finish(rten_status st) {
    if (st == RTEN_OK) {
        for (auto& cb : copybacks) {
            if (cb.bytes) {
                cudaError_t e = cudaMemcpyAsync(cb.host, cb.dev, cb.bytes, cudaMemcpyDeviceToHost, ctx->stream);
                if (e != cudaSuccess) st = fail_cuda(ctx, e, "cudaMemcpyAsync(D2H)");
            }
        }
    } else {
        // give back outputs we allocated for a failed op
        for (rten_tensor* o : allocated) {
            pool_free(ctx, o->data);
            o->data = nullptr;
        }
    }
    release_temps(ctx);
    if (host_involved && !ctx->capturing) {
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess && st == RTEN_OK) st = fail_cuda(ctx, e, "cudaStreamSynchronize");
    }
    return st;
}

}  // namespace rtb

using namespace rtb;

// =========================================================================================
extern "C" {

const char* rten_b200_version(void) { return "rten-b200 0.1 (sm_100a)"; }

// Measured launch plans can be kept across processes: RTEN_B200_TUNE_FILE names a text file that is read when a
// context is created and rewritten when a context that measured new plans is destroyed (one line per problem:
// key integers, '|', plan integers).
static void tune_cache_load(rten_ctx* ctx, const char* path) {
    FILE* f = fopen(path, "r");
    if (!f) return;
    char line[2048];
    while (fgets(line, sizeof(line), f)) {
        std::vector<long long> key;
        std::array<int, 8> plan{};
        char* p = line;
        bool in_plan = false;
        int np = 0;
        while (*p) {
            while (*p == ' ') p++;
            if (*p == '|') {
                in_plan = true;
                p++;
                continue;
            }
            if (*p == '\n' || *p == 0) break;
            char* end = nullptr;
            const long long v = strtoll(p, &end, 10);
            if (end == p) break;
            if (in_plan) {
                if (np < 8) plan[np++] = (int)v;
            } else {
                key.push_back(v);
            }
            p = end;
        }
        if (np == 8 && !key.empty()) ctx->tune_cache[key] = plan;
    }
    fclose(f);
}

static void tune_cache_save(rten_ctx* ctx, const char* path) {
    FILE* f = fopen(path, "w");
    if (!f) return;
    for (const auto& kv : ctx->tune_cache) {
        for (long long v : kv.first) fprintf(f, "%lld ", v);
        fprintf(f, "|");
        for (int v : kv.second) fprintf(f, " %d", v);
        fprintf(f, "\n");
    }
    fclose(f);
}

rten_status rten_b200_ctx_create(int device, void* cuda_stream_or_null, size_t workspace_bytes, rten_ctx** out) {
    if (!out) return RTEN_ERR_INVALID_VALUE;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || device < 0 || device >= count) return RTEN_ERR_CUDA;
    if (cudaSetDevice(device) != cudaSuccess) return RTEN_ERR_CUDA;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return RTEN_ERR_CUDA;
    if (prop.major != 10) return RTEN_ERR_CUDA;  // sm_100a kernels only: no fallback path exists
    rten_ctx* ctx = new rten_ctx();
    ctx->device = device;
    ctx->num_sms = prop.multiProcessorCount;
    if (cuda_stream_or_null) {
        ctx->stream = reinterpret_cast<cudaStream_t>(cuda_stream_or_null);
    } else {
        if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete ctx;
            return RTEN_ERR_CUDA;
        }
        ctx->own_stream = true;
    }
    if (const char* at = getenv("RTEN_B200_AUTOTUNE")) ctx->autotune = atoi(at) != 0;
    if (const char* tf = getenv("RTEN_B200_TUNE_FILE")) {
        tune_cache_load(ctx, tf);
        ctx->tune_loaded = ctx->tune_cache.size();
    }
    const char* mode = getenv("RTEN_B200_F32_MODE");  // default: tf32x3 (fp32-grade); "tf32" opts in to the single pass
    if (mode && strcmp(mode, "tf32x3") == 0) ctx->f32_mode = RTEN_F32_TF32X3;
    if (mode && strcmp(mode, "tf32") == 0) ctx->f32_mode = RTEN_F32_TF32;
    if (workspace_bytes) {  // pre-reserve one pool bucket so the first ops do not pay cudaMalloc
        void* p = nullptr;
        if (pool_alloc(ctx, workspace_bytes, &p) == RTEN_OK) pool_free(ctx, p);
    }
    *out = ctx;
    return RTEN_OK;
}

void rten_b200_ctx_destroy(rten_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto& kv : ctx->pool.free_buckets)
        for (void* p : kv.second) cudaFree(p);
    for (auto& kv : ctx->pool.live) cudaFree(kv.first);
    for (auto& kv : ctx->pool.cap_free)
        for (void* p : kv.second) cudaFree(p);
    for (rten_graph* g : ctx->graphs) {  // graphs that outlive the context keep nothing of it
        for (auto& pb : g->held) cudaFree(pb.first);
        g->held.clear();
        g->ctx = nullptr;
    }
    if (const char* tf = getenv("RTEN_B200_TUNE_FILE"))
        if (ctx->tune_cache.size() > ctx->tune_loaded) tune_cache_save(ctx, tf);
    if (ctx->sk_counters) cudaFree(ctx->sk_counters);
    if (ctx->attn_cnt) cudaFree(ctx->attn_cnt);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char* rten_b200_last_error(rten_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

rten_status rten_b200_sync(rten_ctx* ctx) {
    if (!ctx) return RTEN_ERR_INVALID_VALUE;
    RTB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return RTEN_OK;
}

rten_status rten_b200_set_f32_mode(rten_ctx* ctx, int mode) {
    if (!ctx) return RTEN_ERR_INVALID_VALUE;
    if (mode != RTEN_F32_TF32 && mode != RTEN_F32_TF32X3) return fail(ctx, RTEN_ERR_INVALID_VALUE, "unknown f32 mode");
    ctx->f32_mode = mode;
    return RTEN_OK;
}

rten_status rten_b200_save_plans(rten_ctx* ctx, const char* path) {
    if (!ctx || !path) return RTEN_ERR_INVALID_VALUE;
    tune_cache_save(ctx, path);
    return RTEN_OK;
}
rten_status rten_b200_load_plans(rten_ctx* ctx, const char* path) {
    if (!ctx || !path) return RTEN_ERR_INVALID_VALUE;
    tune_cache_load(ctx, path);
    return RTEN_OK;
}

rten_status rten_b200_set_autotune(rten_ctx* ctx, int enable) {
    if (!ctx) return RTEN_ERR_INVALID_VALUE;
    ctx->autotune = enable != 0;
    return RTEN_OK;
}

rten_status rten_b200_alloc(rten_ctx* ctx, size_t bytes, void** dev_ptr) {
    if (!ctx || !dev_ptr) return RTEN_ERR_INVALID_VALUE;
    cudaSetDevice(ctx->device);
    return pool_alloc(ctx, bytes, dev_ptr);
}
rten_status rten_b200_free(rten_ctx* ctx, void* dev_ptr) {
    if (!ctx) return RTEN_ERR_INVALID_VALUE;
    return pool_free(ctx, dev_ptr);
}
rten_status rten_b200_host_alloc(rten_ctx* ctx, size_t bytes, void** host_ptr) {
    if (!ctx || !host_ptr) return RTEN_ERR_INVALID_VALUE;
    RTB_CUDA(ctx, cudaHostAlloc(host_ptr, bytes ? bytes : 16, cudaHostAllocDefault));
    return RTEN_OK;
}
rten_status rten_b200_host_free(rten_ctx* ctx, void* host_ptr) {
    if (!ctx) return RTEN_ERR_INVALID_VALUE;
    RTB_CUDA(ctx, cudaFreeHost(host_ptr));
    return RTEN_OK;
}

uint64_t rten_b200_launch_count(rten_ctx* ctx) { return ctx ? ctx->launches : 0; }

rten_status rten_b200_debug_forced_plans(rten_ctx* ctx, uint64_t* matched, uint64_t* unmatched) {
    if (!ctx) return RTEN_ERR_INVALID_VALUE;
    if (matched) *matched = ctx->forced_hits;
    if (unmatched) *unmatched = ctx->forced_misses;
    return RTEN_OK;
}

rten_status rten_b200_copy(rten_ctx* ctx, const rten_tensor* src, rten_tensor* dst) {
    if (!ctx || !src || !dst) return RTEN_ERR_INVALID_VALUE;
    cudaSetDevice(ctx->device);
    if (src->ndim != dst->ndim || src->dtype != dst->dtype)
        return fail(ctx, RTEN_ERR_INCOMPATIBLE_SHAPES, "copy: shape or type mismatch");
    for (int i = 0; i < src->ndim; i++)
        if (src->shape[i] != dst->shape[i]) return fail(ctx, RTEN_ERR_INCOMPATIBLE_SHAPES, "copy: shape or type mismatch");
    const int es = dtype_size(src->dtype);
    const size_t bytes = (size_t)numel(src) * es;
    // fast paths: both contiguous
    if (is_contiguous(src) && is_contiguous(dst)) {
        if (!bytes) return RTEN_OK;
        cudaMemcpyKind kind = src->device < 0 ? (dst->device < 0 ? cudaMemcpyHostToHost : cudaMemcpyHostToDevice)
                                              : (dst->device < 0 ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice);
        RTB_CUDA(ctx, cudaMemcpyAsync(dst->data, src->data, bytes, kind, ctx->stream));
        if ((src->device < 0 || dst->device < 0) && !ctx->capturing) RTB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        return RTEN_OK;
    }
    OpScope sc(ctx);
    rten_tensor s, d;
    rten_status st = sc.in(src, &s);
    if (st == RTEN_OK) {
        if (dst->device >= 0) {
            d = *dst;
        } else {
            rten_tensor tmp = *dst;  // host dst (must be contiguous) via temp
            st = sc.out(&tmp, dst->dtype, dst->ndim, dst->shape, &d, nullptr);
        }
    }
    if (st == RTEN_OK) {
        long long shape[RTEN_MAX_DIMS], ss[RTEN_MAX_DIMS], ds[RTEN_MAX_DIMS];
        for (int i = 0; i < s.ndim; i++) {
            shape[i] = s.shape[i];
            ss[i] = s.strides[i];
            ds[i] = d.strides[i];
        }
        st = launch_nd_copy(ctx, es, s.data, d.data, s.ndim, shape, ss, ds);
    }
    return sc.finish(st);
}

// ---- debug: in-kernel pipeline trace of CTA 0 of the GEMM kernel (clock64 at stage hand-offs)
rten_status rten_b200_debug_trace(rten_ctx* ctx, int enable, int64_t* host_out_8192_or_null) {
    if (!ctx) return RTEN_ERR_INVALID_VALUE;
    cudaSetDevice(ctx->device);
    const size_t bytes = 4 * 2048 * sizeof(int64_t);
    if (ctx->trace && host_out_8192_or_null) {
        RTB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        RTB_CUDA(ctx, cudaMemcpy(host_out_8192_or_null, ctx->trace, bytes, cudaMemcpyDeviceToHost));
    }
    if (enable) {
        if (!ctx->trace) RTB_CUDA(ctx, cudaMalloc(&ctx->trace, bytes));
        RTB_CUDA(ctx, cudaMemsetAsync(ctx->trace, 0, bytes, ctx->stream));
    } else if (ctx->trace) {
        cudaFree(ctx->trace);
        ctx->trace = nullptr;
    }
    return RTEN_OK;
}

// ---- CUDA graphs --------------------------------------------------------------------------
rten_status rten_b200_graph_begin(rten_ctx* ctx) {
    if (!ctx) return RTEN_ERR_INVALID_VALUE;
    if (ctx->capturing) return fail(ctx, RTEN_ERR_INVALID_VALUE, "graph capture already active");
    cudaSetDevice(ctx->device);
    RTB_CUDA(ctx, cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeRelaxed));
    ctx->capturing = true;
    ctx->capture_start_launches = ctx->launches;
    return RTEN_OK;
}
rten_status rten_b200_graph_end(rten_ctx* ctx, rten_graph** out) {
    if (!ctx || !out) return RTEN_ERR_INVALID_VALUE;
    if (!ctx->capturing) return fail(ctx, RTEN_ERR_INVALID_VALUE, "no graph capture active");
    ctx->capturing = false;
    rten_graph* g = new rten_graph();
    cudaError_t e = cudaStreamEndCapture(ctx->stream, &g->graph);
    if (e == cudaSuccess) e = cudaGraphInstantiate(&g->exec, g->graph, 0);
    if (e != cudaSuccess) {
        if (g->graph) cudaGraphDestroy(g->graph);
        delete g;
        capture_settle(ctx, nullptr);
        return fail_cuda(ctx, e, "graph capture/instantiate");
    }
    g->ctx = ctx;
    ctx->graphs.push_back(g);
    capture_settle(ctx, g);
    g->kernels = ctx->launches - ctx->capture_start_launches;
    ctx->launches = ctx->capture_start_launches;  // captured launches did not execute
    *out = g;
    return RTEN_OK;
}
rten_status rten_b200_graph_launch(rten_ctx* ctx, rten_graph* g) {
    if (!ctx || !g) return RTEN_ERR_INVALID_VALUE;
    RTB_CUDA(ctx, cudaGraphLaunch(g->exec, ctx->stream));
    ctx->launches += g->kernels;
    return RTEN_OK;
}
void rten_b200_graph_destroy(rten_graph* g) {
    if (!g) return;
    if (g->exec) cudaGraphExecDestroy(g->exec);
    if (g->graph) cudaGraphDestroy(g->graph);
    if (rten_ctx* ctx = g->ctx) {
        // no replay can touch them any more: the parked buffers return to the pool, pinned ones become ordinary again.
        // (Replays still in flight are ordered before any later use: the pool is stream-ordered on the same stream.)
        for (auto& pb : g->held) ctx->pool.free_buckets[pb.second].push_back(pb.first);
        for (auto it = ctx->pool.pinned.begin(); it != ctx->pool.pinned.end();)
            it = it->second == g ? ctx->pool.pinned.erase(it) : std::next(it);
        ctx->graphs.erase(std::remove(ctx->graphs.begin(), ctx->graphs.end(), g), ctx->graphs.end());
    }
    delete g;
}

}  // extern "C"
