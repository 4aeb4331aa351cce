// context.cu — ctx lifetime, error channel, NCCL plumbing (dlopen'd), scalar-pack finish.
#include <dlfcn.h>
#include <nccl.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include "internal.cuh"
#include "reduce.cuh"

// ------------------------------------------------------------------ error channel
static thread_local char g_err[1024] = "";
void cgo_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
extern "C" const char *cgo_last_error(void) { return g_err; }
extern "C" int cgo_version(void) { return 100; }

// ------------------------------------------------------------------ live contexts
// Host languages with garbage collection may finalise a state or an objective AFTER its ctx
// (interpreter shutdown, test fixtures): handles check before they touch the ctx.
#include <mutex>
#include <set>
static std::mutex g_live_mu;
static std::set<cgo_ctx *> g_live;
static void live_add(cgo_ctx *c) { std::lock_guard<std::mutex> l(g_live_mu); g_live.insert(c); }
static void live_remove(cgo_ctx *c) { std::lock_guard<std::mutex> l(g_live_mu); g_live.erase(c); }
bool cgo_ctx_alive(cgo_ctx *c) { std::lock_guard<std::mutex> l(g_live_mu); return g_live.count(c) != 0; }

// ------------------------------------------------------------------ NCCL via dlopen
struct NcclApi {
    void *handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;
static int nccl_load() {
    if (g_nccl.handle) return 0;
    void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    CGO_CHECK(h != nullptr, "dlopen(libnccl.so.2) failed: %s", dlerror());
#define L(name)                                                         \
    *(void **)(&g_nccl.name) = dlsym(h, "nccl" #name);                  \
    CGO_CHECK(g_nccl.name != nullptr, "dlsym(nccl" #name ") failed")
    L(GetUniqueId); L(CommInitRank); L(CommDestroy); L(AllGather); L(AllReduce); L(Send); L(Recv);
    L(GroupStart); L(GroupEnd); L(GetErrorString);
#undef L
    g_nccl.handle = h;
    return 0;
}
#define CGO_NCCL(call)                                                                          \
    do {                                                                                        \
        ncclResult_t r__ = (call);                                                              \
        if (r__ != ncclSuccess) {                                                               \
            cgo_set_error("%s failed: %s", #call, g_nccl.GetErrorString(r__));                  \
            return 3;                                                                           \
        }                                                                                       \
    } while (0)

// ------------------------------------------------------------------ ctx
extern "C" int cgo_ctx_create(int device, void *cuda_stream, cgo_ctx **out) {
    CGO_CHECK(out != nullptr, "cgo_ctx_create: out is NULL");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cgo_set_error("cgo_ctx_create: no CUDA device (%s); libcgoptim has no CPU fallback",
                      cudaGetErrorString(e));
        return 1;
    }
    CGO_CHECK(device >= 0 && device < ndev, "cgo_ctx_create: device %d out of range [0,%d)", device, ndev);
    CGO_CUDA(cudaSetDevice(device));
    cgo_ctx *c = new cgo_ctx();
    c->device = device;
    cudaDeviceProp prop;
    CGO_CUDA(cudaGetDeviceProperties(&prop, device));
    c->sms = prop.multiProcessorCount;
    if (const char *e = getenv("CGO_CSR_MODE")) c->csr_mode = atoi(e);
    if (cuda_stream) {
        c->stream = (cudaStream_t)cuda_stream;
    } else {
        CGO_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        c->own_stream = true;
    }
    CGO_CUDA(cudaMalloc(&c->d_partial, sizeof(double) * CGO_MAXK * CGO_GMAX));
    CGO_CUDA(cudaMalloc(&c->d_ticket, sizeof(unsigned int) * 4));
    CGO_CUDA(cudaMemsetAsync(c->d_ticket, 0, sizeof(unsigned int) * 4, c->stream));
    CGO_CUDA(cudaMalloc(&c->d_progress, sizeof(unsigned long long) * 8));
    CGO_CUDA(cudaMemsetAsync(c->d_progress, 0, sizeof(unsigned long long) * 8, c->stream));
    CGO_CUDA(cudaHostAlloc(&c->h_pack, sizeof(double) * CGO_PACK_LEN, cudaHostAllocMapped));
    CGO_CUDA(cudaHostGetDevicePointer(&c->d_pack_map, c->h_pack, 0));
    CGO_CUDA(cudaMalloc(&c->d_pack, sizeof(double) * CGO_PACK_LEN));
    CGO_CUDA(cudaMalloc(&c->d_scal, sizeof(double) * CGO_NSCAL));
    CGO_CUDA(cudaMemsetAsync(c->d_pack, 0, sizeof(double) * CGO_PACK_LEN, c->stream));
    CGO_CUDA(cudaMemsetAsync(c->d_scal, 0, sizeof(double) * CGO_NSCAL, c->stream));
    CGO_CUDA(cudaStreamSynchronize(c->stream));
    live_add(c);
    *out = c;
    return 0;
}

extern "C" int cgo_ctx_destroy(cgo_ctx *c) {
    if (!c || !cgo_ctx_alive(c)) return 0;
    live_remove(c);
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    if (c->gather_local) cgo_peer_free(c, c->gather_local, c->gather_peer, false);
    if (c->flags_local) cgo_peer_free(c, c->flags_local, c->flags_peer, false);   // teardown: no collective
    cudaFree(c->d_gather_peer); cudaFree(c->d_flags_peer);
    if (c->comm && g_nccl.handle) g_nccl.CommDestroy((ncclComm_t)c->comm);
    cudaFree(c->d_partial); cudaFree(c->d_ticket); cudaFreeHost(c->h_pack);
    cudaFree(c->d_progress);
    cudaFree(c->d_pack); cudaFree(c->d_gather); cudaFree(c->d_scal);
    for (auto &kv : c->dev_pool) for (void *p : kv.second) cudaFree(p);
    for (auto e : c->ev_pool) cudaEventDestroy(e);
    for (auto &t : c->pending) { cudaEventDestroy(t.e0); cudaEventDestroy(t.e1); }
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
    return 0;
}
extern "C" int cgo_ctx_stream(cgo_ctx *c, void **s) {
    CGO_CHECK(c && s, "cgo_ctx_stream: NULL argument");
    *s = (void *)c->stream;
    return 0;
}
extern "C" int cgo_ctx_set_reduction_ctas(cgo_ctx *c, int G) {
    CGO_CHECK(c != nullptr, "NULL ctx");
    CGO_CHECK(G >= 1 && G <= CGO_GMAX, "cgo_ctx_set_reduction_ctas: G=%d out of [1,%d]", G, CGO_GMAX);
    c->G = G;
    return 0;
}
extern "C" int cgo_ctx_set_gather_block_bytes(cgo_ctx *c, int64_t bytes) {
    CGO_CHECK(c != nullptr, "NULL ctx");
    CGO_CHECK(bytes >= 0, "cgo_ctx_set_gather_block_bytes: negative size");
    c->gather_block_bytes = (size_t)bytes;
    return 0;
}
extern "C" int cgo_ctx_sm_count(cgo_ctx *c, int *sms) {
    CGO_CHECK(c && sms, "NULL argument");
    *sms = c->sms;
    return 0;
}
extern "C" int cgo_ctx_set_csr_mode(cgo_ctx *c, int mode) {
    CGO_CHECK(c != nullptr, "NULL ctx");
    CGO_CHECK(mode >= 0 && mode <= 2, "cgo_ctx_set_csr_mode: mode %d out of [0,2]", mode);
    c->csr_mode = mode;
    return 0;
}
extern "C" int cgo_ctx_kernel_launches(cgo_ctx *c, int64_t *count) {
    CGO_CHECK(c && count, "NULL argument");
    *count = c->launches;
    return 0;
}

extern "C" int cgo_comm_get_unique_id(void *id128) {
    CGO_CHECK(id128 != nullptr, "NULL id");
    CGO_TRY(nccl_load());
    ncclUniqueId id;
    CGO_NCCL(g_nccl.GetUniqueId(&id));
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    memcpy(id128, &id, 128);
    return 0;
}
extern "C" int cgo_ctx_comm_init(cgo_ctx *c, int nranks, int rank, const void *id128) {
    CGO_CHECK(c && id128, "NULL argument");
    CGO_CHECK(nranks >= 1 && rank >= 0 && rank < nranks, "bad rank %d / %d", rank, nranks);
    CGO_CUDA(cudaSetDevice(c->device));
    c->nranks = nranks;
    c->rank = rank;
    if (nranks == 1) return 0;
    CGO_TRY(nccl_load());
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    ncclComm_t comm;
    CGO_NCCL(g_nccl.CommInitRank(&comm, nranks, id, rank));
    c->comm = (void *)comm;
    c->nccl = &g_nccl;
    CGO_CUDA(cudaMalloc(&c->d_gather, sizeof(double) * CGO_PACK_LEN * nranks));
    // peer memory: every rank maps every other rank's flag block (CUDA IPC; one node).  When the
    // mapping is refused (no P2P route, IPC disabled, CGO_NO_PEER=1) the halo exchanges stay on
    // NCCL point-to-point transfers.
    const char *no_peer = getenv("CGO_NO_PEER");
    void *fl = nullptr;
    c->peer_ok = true;
    int rc = (no_peer && no_peer[0] == '1') ? 4 : cgo_peer_alloc(c, sizeof(unsigned long long) * CGO_F_N, &fl, c->flags_peer);
    c->flags_local = (unsigned long long *)fl;
    // every rank must take the same path: agree through the communicator
    double ok = (rc == 0) ? 1.0 : 0.0, *d_ok = c->d_scal + CGO_NSCAL - 2;
    CGO_CUDA(cudaMemcpyAsync(d_ok, &ok, sizeof(double), cudaMemcpyHostToDevice, c->stream));
    CGO_NCCL(g_nccl.AllReduce(d_ok, d_ok, 1, ncclFloat64, ncclMin, comm, c->stream));
    CGO_CUDA(cudaMemcpyAsync(&ok, d_ok, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CGO_CUDA(cudaStreamSynchronize(c->stream));
    c->peer_ok = ok > 0.5;
    if (c->peer_ok) {
        CGO_CHECK(nranks <= CGO_MAX_RANKS, "at most %d ranks", CGO_MAX_RANKS);
        void *gl = nullptr;
        CGO_TRY(cgo_peer_alloc(c, sizeof(double) * 2 * (size_t)nranks * CGO_PACK_LEN, &gl, c->gather_peer));
        c->gather_local = (double *)gl;
        CGO_CUDA(cudaMalloc(&c->d_gather_peer, sizeof(void *) * (size_t)nranks));
        CGO_CUDA(cudaMalloc(&c->d_flags_peer, sizeof(void *) * (size_t)nranks));
        CGO_CUDA(cudaMemcpy(c->d_gather_peer, c->gather_peer.data(), sizeof(void *) * (size_t)nranks, cudaMemcpyHostToDevice));
        CGO_CUDA(cudaMemcpy(c->d_flags_peer, c->flags_peer.data(), sizeof(void *) * (size_t)nranks, cudaMemcpyHostToDevice));
        CGO_TRY(cgo_ctx_barrier(c));
    }
    return 0;
}
extern "C" int cgo_ctx_peer_memory(cgo_ctx *c, int *enabled) {
    CGO_CHECK(c && enabled, "NULL argument");
    *enabled = (c->nranks > 1 && c->peer_ok) ? 1 : 0;
    return 0;
}

// ------------------------------------------------------------------ pooled device blocks
int cgo_dev_alloc(cgo_ctx *c, size_t bytes, void **out) {
    auto it = c->dev_pool.find(bytes);
    if (it != c->dev_pool.end() && !it->second.empty()) {
        *out = it->second.back();
        it->second.pop_back();
        c->dev_pool_bytes -= bytes;
    } else {
        CGO_CUDA(cudaMalloc(out, bytes));
    }
    CGO_CUDA(cudaMemsetAsync(*out, 0, bytes, c->stream));
    return 0;
}
void cgo_dev_free(cgo_ctx *c, void *ptr, size_t bytes) {
    if (!ptr) return;
    if (!cgo_ctx_alive(c)) { cudaFree(ptr); return; }
    if (c->dev_pool_bytes + bytes <= ((size_t)24 << 30)) {      // keep at most 24 GB around
        c->dev_pool[bytes].push_back(ptr);
        c->dev_pool_bytes += bytes;
    } else {
        cudaFree(ptr);
    }
}

// release the device blocks the ctx keeps for reuse (up to 24 GB of state vectors of destroyed states); peer-mapped
// blocks stay pooled (freeing them is a collective)
extern "C" int cgo_ctx_trim_pools(cgo_ctx *c, int64_t *freed_bytes) {
    CGO_CHECK(c != nullptr, "NULL ctx");
    CGO_CUDA(cudaSetDevice(c->device));
    CGO_CUDA(cudaStreamSynchronize(c->stream));
    int64_t freed = 0;
    for (auto &kv : c->dev_pool) {
        for (void *p : kv.second) { cudaFree(p); freed += (int64_t)kv.first; }
        kv.second.clear();
    }
    c->dev_pool.clear();
    c->dev_pool_bytes = 0;
    if (freed_bytes) *freed_bytes = freed;
    return 0;
}

// ------------------------------------------------------------------ peer memory (CUDA IPC)
int cgo_peer_alloc(cgo_ctx *c, size_t bytes, void **local, std::vector<void *> &peers) {
    const int R = c->nranks;
    *local = nullptr;
    // a block of this size released earlier (every rank pools in lockstep): mapping a peer's
    // allocation costs milliseconds, so the state vectors of successive runs reuse their blocks
    auto it = c->peer_pool.find(bytes);
    if (it != c->peer_pool.end() && !it->second.empty()) {
        peers = it->second.back();
        it->second.pop_back();
        c->peer_pool_bytes -= bytes;
        *local = peers[(size_t)c->rank];
        CGO_CUDA(cudaMemsetAsync(*local, 0, bytes, c->stream));
        return cgo_ctx_barrier(c);       // no neighbour writes into the block before it is cleared
    }
    peers.assign((size_t)R, nullptr);
    CGO_CUDA(cudaMalloc(local, bytes));
    CGO_CUDA(cudaMemsetAsync(*local, 0, bytes, c->stream));
    peers[(size_t)c->rank] = *local;
    if (R == 1) { c->peer_bytes[*local] = bytes; return 0; }
    CGO_CHECK(c->peer_ok, "peer memory is not available on this communicator");
    cudaIpcMemHandle_t mine;
    CGO_CUDA(cudaIpcGetMemHandle(&mine, *local));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    unsigned char *d_h = nullptr;
    std::vector<cudaIpcMemHandle_t> all((size_t)R);
    int rc = 0;
    auto body = [&]() -> int {
        CGO_CUDA(cudaMalloc(&d_h, 64 * (size_t)(R + 1)));
        CGO_CUDA(cudaMemcpyAsync(d_h + 64 * (size_t)R, &mine, 64, cudaMemcpyHostToDevice, c->stream));
        CGO_NCCL(g_nccl.AllGather(d_h + 64 * (size_t)R, d_h, 64, ncclInt8, (ncclComm_t)c->comm, c->stream));
        CGO_CUDA(cudaMemcpyAsync(all.data(), d_h, 64 * (size_t)R, cudaMemcpyDeviceToHost, c->stream));
        CGO_CUDA(cudaStreamSynchronize(c->stream));
        return 0;
    };
    rc = body();
    cudaFree(d_h);
    if (rc) return rc;
    for (int r = 0; r < R; ++r) {
        if (r == c->rank) continue;
        cudaError_t e = cudaIpcOpenMemHandle(&peers[(size_t)r], all[(size_t)r], cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cgo_set_error("cudaIpcOpenMemHandle(rank %d) failed: %s", r, cudaGetErrorString(e));
            cudaGetLastError();
            return 1;
        }
    }
    c->peer_bytes[*local] = bytes;
    return 0;
}
int cgo_peer_free(cgo_ctx *c, void *local, std::vector<void *> &peers, bool collective) {
    if (!local) return 0;
    if (!cgo_ctx_alive(c)) { peers.clear(); return 0; }      // the ctx went first: the block dies with the process
    if (c->nranks > 1 && collective && peers.size() == (size_t)c->nranks) {
        // keep the block and its mappings for the next allocation of this size; the barrier makes
        // sure no rank still reads or writes it on behalf of the old owner
        size_t bytes = 0;
        auto f = c->peer_bytes.find(local);
        if (f != c->peer_bytes.end()) bytes = f->second;
        if (bytes && c->peer_pool_bytes + bytes <= ((size_t)16 << 30)) {
            cgo_ctx_barrier(c);
            c->peer_pool[bytes].push_back(peers);
            c->peer_pool_bytes += bytes;
            peers.clear();
            return 0;
        }
        // pool full: unmap on every rank, then the owner frees
        cgo_ctx_barrier(c);
        for (int r = 0; r < c->nranks; ++r)
            if (r != c->rank && peers[(size_t)r]) cudaIpcCloseMemHandle(peers[(size_t)r]);
        cgo_ctx_barrier(c);
        c->peer_bytes.erase(local);
        cudaFree(local);
        peers.clear();
        return 0;
    }
    if (c->nranks == 1 && collective) {
        c->peer_bytes.erase(local);
        cudaFree(local);
        peers.clear();
        return 0;
    }
    // teardown (or an incomplete mapping): mappings and blocks die with the process
    peers.clear();
    return 0;
}

extern "C" int cgo_host_alloc(size_t bytes, void **out) {
    CGO_CHECK(out != nullptr, "NULL argument");
    CGO_CUDA(cudaHostAlloc(out, bytes > 0 ? bytes : 1, cudaHostAllocDefault));
    return 0;
}
extern "C" int cgo_host_free(void *ptr) {
    if (ptr) CGO_CUDA(cudaFreeHost(ptr));
    return 0;
}

extern "C" int cgo_shard_range(int64_t n, int nranks, int rank, int64_t align, int64_t *lo, int64_t *hi) {
    CGO_CHECK(lo && hi && nranks >= 1 && rank >= 0 && rank < nranks && align >= 1, "cgo_shard_range: bad arguments");
    int64_t units = n / align;
    *lo = (units * rank / nranks) * align;
    *hi = (rank == nranks - 1) ? n : (units * (rank + 1) / nranks) * align;
    return 0;
}

// ring halo exchange: my head goes to the previous rank (its right halo), my tail to the next
// rank (its left halo)
int cgo_sendrecv_ring(cgo_ctx *c, const double *send_to_prev, double *recv_from_next,
                      const double *send_to_next, double *recv_from_prev, int64_t count) {
    if (count <= 0) return 0;
    if (c->nranks == 1) {
        CGO_CUDA(cudaMemcpyAsync(recv_from_next, send_to_prev, sizeof(double) * count, cudaMemcpyDeviceToDevice, c->stream));
        CGO_CUDA(cudaMemcpyAsync(recv_from_prev, send_to_next, sizeof(double) * count, cudaMemcpyDeviceToDevice, c->stream));
        return 0;
    }
    int prev = (c->rank + c->nranks - 1) % c->nranks, next = (c->rank + 1) % c->nranks;
    ncclComm_t comm = (ncclComm_t)c->comm;
    CGO_NCCL(g_nccl.GroupStart());
    CGO_NCCL(g_nccl.Send(send_to_prev, (size_t)count, ncclFloat64, prev, comm, c->stream));
    CGO_NCCL(g_nccl.Recv(recv_from_next, (size_t)count, ncclFloat64, next, comm, c->stream));
    CGO_NCCL(g_nccl.Send(send_to_next, (size_t)count, ncclFloat64, next, comm, c->stream));
    CGO_NCCL(g_nccl.Recv(recv_from_prev, (size_t)count, ncclFloat64, prev, comm, c->stream));
    CGO_NCCL(g_nccl.GroupEnd());
    return 0;
}

// all-gather of unequal contiguous shards: rank r owns [lo[r], lo[r+1]) of `full`; its own
// shard is copied in from `mine`.  Grouped point-to-point transfers (NVLink through NVSwitch).
int cgo_allgatherv_f64(cgo_ctx *c, const double *mine, double *full, const int64_t *lo) {
    const int R = c->nranks, me = c->rank;
    const int64_t cnt = lo[me + 1] - lo[me];
    if (cnt > 0 && full + lo[me] != mine)
        CGO_CUDA(cudaMemcpyAsync(full + lo[me], mine, sizeof(double) * (size_t)cnt, cudaMemcpyDeviceToDevice, c->stream));
    if (R == 1) return 0;
    ncclComm_t comm = (ncclComm_t)c->comm;
    CGO_NCCL(g_nccl.GroupStart());
    for (int k = 1; k < R; ++k) {
        const int to = (me + k) % R, from = (me + R - k) % R;
        if (cnt > 0) CGO_NCCL(g_nccl.Send(mine, (size_t)cnt, ncclFloat64, to, comm, c->stream));
        if (lo[from + 1] > lo[from])
            CGO_NCCL(g_nccl.Recv(full + lo[from], (size_t)(lo[from + 1] - lo[from]), ncclFloat64, from, comm, c->stream));
    }
    CGO_NCCL(g_nccl.GroupEnd());
    return 0;
}

// ------------------------------------------------------------------ per-launch timing
static cudaEvent_t ev_get(cgo_ctx *c) {
    if (!c->ev_pool.empty()) { cudaEvent_t e = c->ev_pool.back(); c->ev_pool.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}
void cgo_timer_begin(cgo_ctx *c, int cls) {
    if (!c->timing) return;
    CgoPendingTimer t;
    t.cls = cls; t.e0 = ev_get(c); t.e1 = ev_get(c);
    cudaEventRecord(t.e0, c->stream);
    c->pending.push_back(t);
}
void cgo_timer_end(cgo_ctx *c) {
    if (!c->timing || c->pending.empty()) return;
    cudaEventRecord(c->pending.back().e1, c->stream);
}
void cgo_timer_collect(cgo_ctx *c) {
    for (auto &t : c->pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, t.e0, t.e1) == cudaSuccess) { c->t_ms[t.cls] += ms; c->t_cnt[t.cls]++; }
        c->ev_pool.push_back(t.e0); c->ev_pool.push_back(t.e1);
    }
    c->pending.clear();
}
extern "C" int cgo_ctx_timing(cgo_ctx *c, int enable) {
    CGO_CHECK(c != nullptr, "NULL ctx");
    CGO_CUDA(cudaStreamSynchronize(c->stream));
    cgo_timer_collect(c);
    c->timing = enable != 0;
    return 0;
}
extern "C" int cgo_ctx_timing_read(cgo_ctx *c, double *ms, int64_t *counts, int reset) {
    CGO_CHECK(c && ms && counts, "NULL argument");
    CGO_CUDA(cudaStreamSynchronize(c->stream));
    cgo_timer_collect(c);
    for (int i = 0; i < CGO_T_N; ++i) { ms[i] = c->t_ms[i]; counts[i] = c->t_cnt[i]; }
    if (reset) for (int i = 0; i < CGO_T_N; ++i) { c->t_ms[i] = 0; c->t_cnt[i] = 0; }
    return 0;
}

// ------------------------------------------------------------------ scalar pack finish
RedArgs cgo_red_args(cgo_ctx *c, int slot) {
    RedArgs r;
    r.partial = c->d_partial;
    r.ticket = c->d_ticket;
    r.out = ((c->nranks > 1) ? c->d_pack : c->d_pack_map) + slot;
    r.G = c->G;
    return r;
}

// shard results are added in rank order on every rank (canonical order, last level)
__global__ void k_sum_ranks(const double *gathered, int nranks, int K, double *out) {
    int k = threadIdx.x;
    if (k < K) {
        double s = gathered[k];
        for (int r = 1; r < nranks; ++r) s = s + gathered[(size_t)r * CGO_PACK_LEN + k];
        out[k] = s;
    }
    __threadfence_system();
}

// All-gather of the scalar pack over peer memory + rank-ordered sum, one small kernel: thread
// (r, k) stores my pack entry k into rank r's gather block, thread r then release-stores my
// flag in rank r's flag block; thread r waits for rank r's flag here, and the first K threads
// add the R packs in rank order.  Double-buffered by the epoch's parity (a fast rank may already
// deliver the next pack while a slow one still sums this one).
__global__ void k_pack_exchange(const double *pack, void *const *gather_peer, void *const *flags_peer,
                                const double *gather_local, const unsigned long long *flags_local,
                                int nranks, int me, int K, unsigned long long epoch, double *out) {
    const int t = threadIdx.x;
    const size_t buf = (size_t)(epoch & 1ULL) * (size_t)nranks * CGO_PACK_LEN;
    for (int i = t; i < nranks * CGO_PACK_LEN; i += blockDim.x) {
        const int r = i / CGO_PACK_LEN, k = i - r * CGO_PACK_LEN;
        double *dst = (double *)gather_peer[r] + buf + (size_t)me * CGO_PACK_LEN + k;
        *dst = k < K ? pack[k] : 0.0;
    }
    __threadfence_system();
    __syncthreads();
    if (t < nranks) {
        cgo_st_release_sys((unsigned long long *)flags_peer[t] + CGO_F_PACK + me, epoch);
        cgo_spin_until(flags_local + CGO_F_PACK + t, epoch);
    }
    __syncthreads();
    if (t < K) {
        const double *g = gather_local + buf;
        double s = __ldcv(g + t);
        for (int r = 1; r < nranks; ++r) s = s + __ldcv(g + (size_t)r * CGO_PACK_LEN + t);
        out[t] = s;
    }
    __threadfence_system();
}
// after the kernels of one sequence wrote their sums to d_pack: combine the ranks' packs into
// `out_dev` (device or mapped host memory) on every rank, in rank order
int cgo_combine_ranks(cgo_ctx *c, int K, double *out_dev) {
    if (c->peer_ok) {
        const unsigned long long e = ++c->pack_epoch;
        k_pack_exchange<<<1, 128, 0, c->stream>>>(c->d_pack, c->d_gather_peer, c->d_flags_peer, c->gather_local,
                                                  c->flags_local, c->nranks, c->rank, K, e, out_dev);
        c->launches++;
        CGO_CUDA(cudaGetLastError());
        return 0;
    }
    CGO_NCCL(g_nccl.AllGather(c->d_pack, c->d_gather, CGO_PACK_LEN, ncclFloat64, (ncclComm_t)c->comm, c->stream));
    k_sum_ranks<<<1, 32, 0, c->stream>>>(c->d_gather, c->nranks, K, out_dev);
    c->launches++;
    return 0;
}

int cgo_finish_pack(cgo_ctx *c, int K, double *out_host) {
    if (c->nranks > 1) CGO_TRY(cgo_combine_ranks(c, K, c->d_pack_map));
    CGO_CUDA(cudaStreamSynchronize(c->stream));
    if (c->timing) cgo_timer_collect(c);
    for (int k = 0; k < K; ++k) out_host[k] = c->h_pack[k];
    return 0;
}

extern "C" int cgo_ctx_barrier(cgo_ctx *c) {
    CGO_CHECK(c != nullptr, "NULL ctx");
    if (c->nranks > 1) {
        CGO_NCCL(g_nccl.AllReduce(c->d_scal + CGO_NSCAL - 1, c->d_scal + CGO_NSCAL - 1, 1, ncclFloat64, ncclSum, (ncclComm_t)c->comm, c->stream));
    }
    CGO_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}
