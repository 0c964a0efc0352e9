// Cross-rank exchange for the batch-sharded int8 path (SURVEY.md 8e): when a batch is split over GPUs, every rank must
// quantise with the min / max of the WHOLE tensor to stay bit-identical to the unsharded reference
// (src/ops/quantize.rs:352-434 computes one range per tensor).  That is an all-reduce of two numbers per
// DynamicQuantizeLinear -- 53 of them per ResNet-50 step, each on the critical path.
//
// Default path: ONE small kernel per exchange over NVLink peer memory.  Every rank owns a mailbox (cudaMalloc, opened
// by the peers through CUDA IPC at comm_create); the kernel stores (epoch, min) and (epoch, max) as two 64-bit words
// into its slot of every peer's mailbox, spins until every slot of its own mailbox carries the current epoch, and
// reduces.  No fences are needed (each word is self-validating), slots are double-buffered by epoch parity (a rank
// can be at most one exchange ahead of a peer), and the epoch lives in device memory so that CUDA-graph replays advance
// it.  Measured against two ncclAllReduce calls of one int each (the fallback, RTEN_B200_NCCL_RANGES=1): DESIGN.md 5.
// NCCL is resolved at run time (dlopen of libnccl.so.2 -- the copy already loaded in the process if there is one), so
// the library itself keeps no link-time dependency on it; it also carries the IPC handles at start-up.
#include <dlfcn.h>

#include <vector>

#include "comm_device.cuh"
#include "common.h"

struct Id128 {  // ncclUniqueId: 128 opaque bytes, passed BY VALUE to ncclCommInitRank
    char bytes[128];
};

using namespace rtb;

namespace {

struct NcclApi {
    void* handle = nullptr;
    int (*GetUniqueId)(void*) = nullptr;
    int (*CommInitRank)(void**, int, Id128, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};

NcclApi g_nccl;

bool load_nccl() {
    if (g_nccl.handle) return true;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW);
    if (!h) return false;
    NcclApi a;
    a.handle = h;
    a.GetUniqueId = reinterpret_cast<decltype(a.GetUniqueId)>(dlsym(h, "ncclGetUniqueId"));
    a.CommInitRank = reinterpret_cast<decltype(a.CommInitRank)>(dlsym(h, "ncclCommInitRank"));
    a.CommDestroy = reinterpret_cast<decltype(a.CommDestroy)>(dlsym(h, "ncclCommDestroy"));
    a.AllReduce = reinterpret_cast<decltype(a.AllReduce)>(dlsym(h, "ncclAllReduce"));
    a.AllGather = reinterpret_cast<decltype(a.AllGather)>(dlsym(h, "ncclAllGather"));
    a.GetErrorString = reinterpret_cast<decltype(a.GetErrorString)>(dlsym(h, "ncclGetErrorString"));
    if (!a.GetUniqueId || !a.CommInitRank || !a.CommDestroy || !a.AllReduce) return false;
    g_nccl = a;
    return true;
}

constexpr int kNcclInt8 = 0;   // ncclInt8 / ncclChar
constexpr int kNcclInt32 = 2;  // ncclInt32
constexpr int kNcclMax = 2;    // ncclMax
constexpr int kNcclMin = 3;    // ncclMin

// mm[0] / mm[1]: ordered-int encodings of the local min / max (integer order == float order)
__global__ void __launch_bounds__(32) peer_minmax_kernel(int* mm, const PeerTable peers, int rank, int world) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    peer_minmax_warp(mm, peers, rank, world);
}

}  // namespace

struct rten_comm {
    void* nccl = nullptr;
    int rank = 0, world = 1;
    Mailbox* box = nullptr;       // local mailbox (cudaMalloc)
    PeerTable peers = {};         // peers' mailboxes opened through CUDA IPC (peer_ok)
    bool peer_ok = false;
};

namespace rtb {

// min / max all-reduce of the two ORDERED-INT encoded floats produced by the local min/max kernel (rowops.cu): integer
// min / max on that encoding is the float min / max, and is exact and order independent.
rten_status comm_allreduce_minmax(rten_ctx* ctx, rten_comm* comm, int* mm) {
    if (!comm || comm->world <= 1) return RTEN_OK;
    cudaStream_t s = ctx->stream;
    if (comm->peer_ok) {
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3(1);
        cfg.blockDim = dim3(32);
        cfg.stream = s;
        cudaLaunchAttribute attr[1];
        fill_launch_attrs(cfg, attr, false);
        cudaError_t e = cudaLaunchKernelEx(&cfg, peer_minmax_kernel, mm, comm->peers, comm->rank, comm->world);
        if (e != cudaSuccess) return fail_cuda(ctx, e, "peer min/max exchange launch");
        count_launch(ctx);
        return RTEN_OK;
    }
    int r = g_nccl.AllReduce(mm, mm, 1, kNcclInt32, kNcclMin, comm->nccl, s);
    if (r == 0) r = g_nccl.AllReduce(mm + 1, mm + 1, 1, kNcclInt32, kNcclMax, comm->nccl, s);
    if (r != 0) {
        ctx->err = std::string("ncclAllReduce failed: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
        return RTEN_ERR_NCCL;
    }
    count_launch(ctx, 2);
    return RTEN_OK;
}

// the quantise kernels run the exchange themselves (rowops.cu): hand them the peer table, or world = 0 when this
// communicator exchanges through NCCL (the caller then takes comm_allreduce_minmax first)
bool comm_range_exchange(rten_comm* comm, RangeExchange* out) {
    memset(out, 0, sizeof(*out));
    if (!comm || comm->world <= 1 || !comm->peer_ok || getenv("RTEN_B200_UNFUSED_RANGE_EXCHANGE")) return false;
    out->peers = comm->peers;
    out->rank = comm->rank;
    out->world = comm->world;
    return true;
}

}  // namespace rtb

// Peer mailboxes: allocate, exchange the IPC handles through NCCL, open the peers'.  Any failure leaves the communicator
// on the NCCL path (peer_ok = false) -- both are exact, the choice only changes the latency.
static void setup_peer_mailboxes(rten_ctx* ctx, rten_comm* c) {
    if (getenv("RTEN_B200_NCCL_RANGES") || c->world > MAX_PEERS || !g_nccl.AllGather) return;
    if (cudaMalloc(&c->box, sizeof(Mailbox)) != cudaSuccess) {
        cudaGetLastError();
        c->box = nullptr;
        return;
    }
    cudaMemset(c->box, 0, sizeof(Mailbox));
    cudaIpcMemHandle_t mine;
    int ok = cudaIpcGetMemHandle(&mine, c->box) == cudaSuccess ? 1 : 0;
    // gather {handle, ok} of every rank (device staging buffers: NCCL moves device memory)
    struct Entry {
        cudaIpcMemHandle_t h;
        int ok;
        int pad[3];
    };
    Entry e_host;
    memset(&e_host, 0, sizeof(e_host));
    e_host.h = mine;
    e_host.ok = ok;
    Entry *d_send = nullptr, *d_recv = nullptr;
    std::vector<Entry> all(c->world);
    bool good = cudaMalloc(&d_send, sizeof(Entry)) == cudaSuccess && cudaMalloc(&d_recv, sizeof(Entry) * c->world) == cudaSuccess;
    if (good) {
        cudaMemcpy(d_send, &e_host, sizeof(Entry), cudaMemcpyHostToDevice);
        cudaStream_t s = ctx->stream;
        good = g_nccl.AllGather(d_send, d_recv, sizeof(Entry), kNcclInt8, c->nccl, s) == 0 && cudaStreamSynchronize(s) == cudaSuccess;
        if (good) cudaMemcpy(all.data(), d_recv, sizeof(Entry) * c->world, cudaMemcpyDeviceToHost);
    }
    if (d_send) cudaFree(d_send);
    if (d_recv) cudaFree(d_recv);
    // every rank must take the same decision: all handles valid, and every open succeeds (second round below)
    int opened = good ? 1 : 0;
    for (int r = 0; r < c->world && opened; r++) opened = all[r].ok;
    for (int r = 0; r < c->world && opened; r++) {
        if (r == c->rank) {
            c->peers.box[r] = c->box;
            continue;
        }
        void* p = nullptr;
        if (cudaIpcOpenMemHandle(&p, all[r].h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
            cudaGetLastError();
            opened = 0;
            break;
        }
        c->peers.box[r] = reinterpret_cast<Mailbox*>(p);
    }
    // agree: min over ranks of `opened` (one int all-reduce; the last NCCL call of the set-up)
    int* d_flag = nullptr;
    if (cudaMalloc(&d_flag, 4) == cudaSuccess) {
        cudaMemcpy(d_flag, &opened, 4, cudaMemcpyHostToDevice);
        if (g_nccl.AllReduce(d_flag, d_flag, 1, kNcclInt32, kNcclMin, c->nccl, ctx->stream) == 0 && cudaStreamSynchronize(ctx->stream) == cudaSuccess)
            cudaMemcpy(&opened, d_flag, 4, cudaMemcpyDeviceToHost);
        else
            opened = 0;
        cudaFree(d_flag);
    } else {
        opened = 0;
    }
    c->peer_ok = opened != 0;
}

extern "C" {

rten_status rten_b200_comm_unique_id(void* id128) {
    if (!id128) return RTEN_ERR_INVALID_VALUE;
    if (!load_nccl()) return RTEN_ERR_NCCL;
    return g_nccl.GetUniqueId(id128) == 0 ? RTEN_OK : RTEN_ERR_NCCL;
}

rten_status rten_b200_comm_create(rten_ctx* ctx, const void* id128, int rank, int world, rten_comm** out) {
    if (!ctx || !id128 || !out || world < 1 || rank < 0 || rank >= world) return RTEN_ERR_INVALID_VALUE;
    *out = nullptr;
    if (!load_nccl()) return rtb::fail(ctx, RTEN_ERR_NCCL, "libnccl.so.2 could not be loaded");
    cudaSetDevice(ctx->device);
    Id128 id;
    memcpy(id.bytes, id128, sizeof(id.bytes));
    rten_comm* c = new rten_comm();
    c->rank = rank;
    c->world = world;
    const int r = g_nccl.CommInitRank(&c->nccl, world, id, rank);
    if (r != 0) {
        ctx->err = std::string("ncclCommInitRank failed: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
        delete c;
        return RTEN_ERR_NCCL;
    }
    setup_peer_mailboxes(ctx, c);
    *out = c;
    return RTEN_OK;
}

int rten_b200_comm_uses_peer_memory(const rten_comm* comm) { return comm && comm->peer_ok ? 1 : 0; }

/* Exchanges that timed out waiting for a peer since comm_create (0 in a healthy run): host read of the local mailbox. */
int rten_b200_comm_timeouts(const rten_comm* comm) {
    if (!comm || !comm->box) return 0;
    unsigned v = 0;
    if (cudaMemcpy(&v, &comm->box->timeouts, 4, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    return (int)v;
}

void rten_b200_comm_destroy(rten_comm* comm) {
    if (!comm) return;
    if (comm->peer_ok)
        for (int r = 0; r < comm->world; r++)
            if (r != comm->rank && comm->peers.box[r]) cudaIpcCloseMemHandle(comm->peers.box[r]);
    if (comm->box) cudaFree(comm->box);
    if (comm->nccl && g_nccl.CommDestroy) g_nccl.CommDestroy(comm->nccl);
    delete comm;
}

}  // extern "C"
