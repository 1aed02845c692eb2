// lkb_core.cu -- context, device abstract_vector / basis objects and abstract_linop objects
// behind the C ABI of include/lkb.h.  No CPU fallback: every entry point needs a CUDA device.
#include <dlfcn.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <memory>
#include "../../include/lkb.h"
#include "lkb_internal.h"

using namespace lkb;

namespace lkb {
static thread_local char g_err[1024] = "";
void set_error(const char* fmt, ...) {
    va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
}

static NcclApi g_nccl;
static bool g_nccl_tried = false;
NcclApi* nccl_api() {
    if (g_nccl.handle) return &g_nccl;
    if (g_nccl_tried) return nullptr;
    g_nccl_tried = true;
    const char* cands[] = { getenv("LKB_NCCL_LIB"), "libnccl.so.2", "libnccl.so",
                            "/usr/local/cuda/lib64/libnccl.so.2", "/usr/lib/x86_64-linux-gnu/libnccl.so.2" };
    void* h = nullptr;
    for (const char* p : cands) { if (!p) continue; h = dlopen(p, RTLD_NOW | RTLD_GLOBAL); if (h) break; }
    if (!h) { set_error("cannot dlopen libnccl (set LKB_NCCL_LIB): %s", dlerror()); return nullptr; }
#define LKB_SYM(field, name) *(void**)(&g_nccl.field) = dlsym(h, name); if (!g_nccl.field) { set_error("missing %s", name); return nullptr; }
    LKB_SYM(GetUniqueId, "ncclGetUniqueId") LKB_SYM(CommInitRank, "ncclCommInitRank") LKB_SYM(CommDestroy, "ncclCommDestroy")
    LKB_SYM(AllReduce, "ncclAllReduce") LKB_SYM(Broadcast, "ncclBroadcast") LKB_SYM(AllGather, "ncclAllGather") LKB_SYM(Reduce, "ncclReduce") LKB_SYM(Send, "ncclSend") LKB_SYM(Recv, "ncclRecv")
    LKB_SYM(GroupStart, "ncclGroupStart") LKB_SYM(GroupEnd, "ncclGroupEnd") LKB_SYM(GetErrorString, "ncclGetErrorString")
#undef LKB_SYM
    g_nccl.handle = h;
    return &g_nccl;
}
int comm_destroy(void* comm) {
    NcclApi* api = nccl_api();
    return api ? api->CommDestroy(comm) : LKB_ERR_NCCL;
}
#define LKB_NCCL(call) do { int r_ = (call); if (r_ != 0) { \
    lkb::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, nccl_api()->GetErrorString(r_)); return LKB_ERR_NCCL; } } while (0)

int check_launch(lkb_ctx_s*, const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("kernel launch failed (%s): %s", what, cudaGetErrorString(e)); return LKB_ERR_CUDA; }
    return 0;
}

void prof_begin(lkb_ctx_s* c, int cls) {
    if (!c->profile || c->capturing) return;
    lkb_ctx_s::ProfEv ev; ev.cls = cls;
    cudaEventCreate(&ev.a); cudaEventCreate(&ev.b);
    cudaEventRecord(ev.a, c->stream);
    c->prof_evs.push_back(ev);
}
void prof_end(lkb_ctx_s* c, int cls, int nlaunch) {
    c->launches += nlaunch;
    if (!c->profile || c->capturing) return;
    cudaEventRecord(c->prof_evs.back().b, c->stream);
    c->prof_n[cls] += nlaunch;
}
int prof_collect(lkb_ctx_s* c) {
    if (c->prof_evs.empty()) return 0;
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    for (auto& ev : c->prof_evs) {
        float ms = 0.f; cudaEventElapsedTime(&ms, ev.a, ev.b);
        c->prof_ms[ev.cls] += ms;
        cudaEventDestroy(ev.a); cudaEventDestroy(ev.b);
    }
    c->prof_evs.clear();
    return 0;
}

// Captured graphs hold raw pointers into the context workspaces and into bases / operators: whenever
// one of those allocations goes away the cached executables that may reference it are dropped.
void invalidate_graphs(lkb_ctx_s* c, uint64_t uid) {
    if (uid == 0) { c->graph_cache.clear(); return; }
    char tag[40]; snprintf(tag, sizeof(tag), ":%llu:", (unsigned long long)uid);
    for (auto it = c->graph_cache.begin(); it != c->graph_cache.end();) {
        if (it->first.find(tag) != std::string::npos) it = c->graph_cache.erase(it);
        else ++it;
    }
}
static int grow(lkb_ctx_s* c, CudaPtr<void>& p, size_t* cur, size_t need) {
    if (*cur >= need) return 0;
    cudaStreamSynchronize(c->stream);
    invalidate_graphs(c, 0);
    p.reset(); *cur = 0;
    LKB_TRY(cuda_alloc(p, need));
    *cur = need;
    return 0;
}
int ensure_ws(lkb_ctx_s* c, int jp) {
    if (c->capturing) return 0;   // sized before capture begins
    const size_t need = (size_t)MAX_ROWBLOCKS * (size_t)jp * 16;
    LKB_TRY(grow(c, c->partial, &c->partial_bytes, std::max(need, (size_t)MAX_ROWBLOCKS * 16 * 8)));
    if (c->cbuf_len < (size_t)jp) {
        size_t len = std::max((size_t)jp, (size_t)272);
        cudaStreamSynchronize(c->stream);
        invalidate_graphs(c, 0);
        c->c1.reset(); c->c2.reset(); c->tmpw.reset(); c->cbuf_len = 0;
        LKB_TRY(cuda_alloc(c->c1, len * 16)); LKB_TRY(cuda_alloc(c->c2, len * 16)); LKB_TRY(cuda_alloc(c->tmpw, len * 16));
        c->cbuf_len = len;
    }
    return 0;
}
int ensure_hstage(lkb_ctx_s* c, size_t bytes) {
    if (c->hstage_bytes >= bytes) return 0;
    c->hstage = nullptr; c->hstage_mem.reset(); c->hstage_bytes = 0;
    LKB_TRY(cuda_alloc(c->hstage_mem, bytes));
    c->hstage = c->hstage_mem; c->hstage_bytes = bytes;
    return 0;
}
int ensure_Hd(lkb_ctx_s* c, size_t bytes) { return grow(c, c->Hd, &c->Hd_bytes, bytes); }
int ensure_coefd(lkb_ctx_s* c, size_t bytes) {
    const int r = grow(c, c->coefd_mem, &c->coefd_bytes, bytes);
    c->coefd = c->coefd_mem;
    return r;
}

int allreduce_w(lkb_ctx_s* c, void* buf, size_t ndoubles) {
    if (c->world == 1 || c->p2p_active) return 0;      // p2p: already reduced inside the producing kernel
    NcclApi* api = nccl_api();
    if (!api) return LKB_ERR_NCCL;
    LKB_NCCL(api->AllReduce(buf, buf, ndoubles, /*ncclFloat64*/ 8, /*ncclSum*/ 0, c->comm, c->stream));
    pdl_rearm();                                       // the next kernel follows an NCCL operation: normal launch
    return 0;
}
int& pdl_state() { static thread_local int s = 0; return s; }
int& sweep_dir() { static thread_local int d = 0; return d; }
// Stream-ordered allocation of vectors / bases / solver work space from the device's default memory pool with an
// unlimited release threshold: freed blocks stay cached in the pool, so the GB-sized work bases that gmres / cg /
// eigs allocate per call (`allocate(V(kdim+1), source=b)` in the reference) cost a pool lookup instead of a
// cudaMalloc / cudaFree pair (measured in round 1: 0.3-1 s of call-to-call variance).  P2P / IPC regions stay on
// cudaMalloc (CUDA IPC handles cannot be taken of pool memory).
int dev_alloc(lkb_ctx_s* c, void** p, size_t bytes) {
    cudaError_t e = cudaMallocAsync(p, bytes ? bytes : 16, c->stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("cudaMallocAsync(%zu) failed: %s", bytes, cudaGetErrorString(e));
        *p = nullptr;
        return LKB_ERR_ALLOC;
    }
    return 0;
}
void dev_free(lkb_ctx_s* c, void* p) {
    if (p) cudaFreeAsync(p, c->stream);      // stream-ordered: no host synchronisation needed
}
static uint64_t g_uid = 0;
uint64_t next_uid() { return ++g_uid; }
// The k x k host algebra (geev / gees+trsen / syev / gesdd) runs redundantly on every rank; a threaded
// LAPACK need not be bitwise reproducible across processes, and a rank that decides "converged" one
// step earlier than its peers would deadlock the collectives.  Rank 0's results are broadcast.
int bcast_host(lkb_ctx_s* c, void* host_buf, size_t bytes) {
    if (c->world == 1 || bytes == 0) return 0;
    NcclApi* api = nccl_api();
    if (!api) return LKB_ERR_NCCL;
    const size_t padded = (bytes + 15) & ~(size_t)15;
    LKB_TRY(ensure_hstage(c, padded + 4096));
    LKB_TRY(ensure_coefd(c, std::max(padded, (size_t)4096)));
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    memcpy(c->hstage, host_buf, bytes);
    LKB_CUDA(cudaMemcpyAsync(c->coefd, c->hstage, padded, cudaMemcpyHostToDevice, c->stream));
    LKB_NCCL(api->Broadcast(c->coefd, c->coefd, padded, /*ncclInt8*/ 0, 0, c->comm, c->stream));
    LKB_CUDA(cudaMemcpyAsync(c->hstage, c->coefd, padded, cudaMemcpyDeviceToHost, c->stream));
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    memcpy(host_buf, c->hstage, bytes);
    return 0;
}
uint64_t next_seed(lkb_ctx_s* c) { return c->seed + 0x9E3779B97F4A7C15ULL * (++c->seed_calls); }

int fetch_flags(lkb_ctx_s* c, int* host_flags) {
    LKB_TRY(ensure_hstage(c, 4096));
    LKB_CUDA(cudaMemcpyAsync(c->hstage, c->flags, F_COUNT * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    memcpy(host_flags, c->hstage, F_COUNT * sizeof(int));
    return 0;
}

int norm2_enqueue(lkb_ctx_s* c, int kind, const void* w, int64_t n, const int* flags) {
    LKB_TRY(ensure_ws(c, 1));
    return dot_reduce(c, kind, w, n, 0, w, n, c->nrm2, flags);
}
int vec_norm_sync(lkb_ctx_s* c, int kind, const void* w, int64_t n, double* out) {
    LKB_TRY(norm2_enqueue(c, kind, w, n, nullptr));
    LKB_TRY(ensure_hstage(c, 4096));
    LKB_CUDA(cudaMemcpyAsync(c->hstage, c->nrm2, 16, cudaMemcpyDeviceToHost, c->stream));
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    *out = sqrt(fabs(*(double*)c->hstage));
    return 0;
}
int vec_dot_sync(lkb_ctx_s* c, int kind, const void* x, const void* y, int64_t n, Scalar* out) {
    LKB_TRY(ensure_ws(c, 2));
    LKB_TRY(dot_reduce(c, kind, x, n, 1, y, n, c->tmpw, nullptr));
    LKB_TRY(ensure_hstage(c, 4096));
    LKB_CUDA(cudaMemcpyAsync(c->hstage, c->tmpw, 16, cudaMemcpyDeviceToHost, c->stream));
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    out->re = ((double*)c->hstage)[0];
    out->im = kind_cplx(kind) ? ((double*)c->hstage)[1] : 0.0;
    return 0;
}
}  // namespace lkb

extern "C" {

const char* lkb_last_error(void) { return g_err; }

int lkb_init(int device, lkb_ctx_t* ctx) { return lkb_init_dist(device, 0, 1, nullptr, ctx); }
int lkb_nccl_unique_id(void* id128) {
    NcclApi* api = nccl_api();
    if (!api) return LKB_ERR_NCCL;
    LKB_NCCL(api->GetUniqueId(id128));
    return 0;
}
int lkb_init_dist(int device, int rank, int world, const void* id128, lkb_ctx_t* ctx) {
    if (!ctx || world < 1 || rank < 0 || rank >= world) return LKB_ERR_ARG;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        set_error("no CUDA device available (%s): liblkb has no CPU fallback", cudaGetErrorString(e));
        return LKB_ERR_CUDA;
    }
    LKB_CUDA(cudaSetDevice(device));
    std::unique_ptr<lkb_ctx_s> c(new lkb_ctx_s());      // a failure below releases what was built so far
    c->dev = device; c->rank = rank; c->world = world;
    LKB_CUDA(cudaDeviceGetAttribute(&c->sms, cudaDevAttrMultiProcessorCount, device));
    LKB_CUDA(cudaStreamCreateWithFlags(c->stream.out(), cudaStreamNonBlocking));
    {   // keep freed blocks in the default pool (see dev_alloc)
        cudaMemPool_t pool = nullptr;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess && pool) {
            unsigned long long thr = ~0ULL;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        }
        cudaGetLastError();
    }
    LKB_TRY(cuda_alloc(c->nrm2, 64));
    LKB_TRY(cuda_alloc(c->inv, 64));
    LKB_TRY(cuda_alloc(c->flags, F_COUNT * sizeof(int)));
    LKB_TRY(cuda_alloc(c->counter, 1024));      // global ticket + one per group of the reduction tree
    LKB_CUDA(cudaMemset(c->flags, 0, F_COUNT * sizeof(int)));
    LKB_CUDA(cudaMemset(c->counter, 0, 1024));
    LKB_CUDA(cudaMemset(c->nrm2, 0, 64));
    LKB_TRY(ensure_ws(c.get(), 272));
    LKB_TRY(ensure_hstage(c.get(), 1 << 20));
    if (world > 1) {
        NcclApi* api = nccl_api();
        if (!api) return LKB_ERR_NCCL;
        NcclId id; memcpy(&id, id128, sizeof(id));
        LKB_NCCL(api->CommInitRank(c->comm.out(), world, id, rank));
    }
    *ctx = c.release();
    return 0;
}
int lkb_finalize(lkb_ctx_t c) {
    if (!c) return LKB_ERR_ARG;
    const int dev = c->dev;
    cudaSetDevice(dev);
    cudaStreamSynchronize(c->stream);
    delete c;
    {
        cudaMemPool_t pool = nullptr;
        if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess && pool) cudaMemPoolTrimTo(pool, 0);
        cudaGetLastError();
    }
    return 0;
}
int lkb_sync(lkb_ctx_t c) { LKB_CUDA(cudaStreamSynchronize(c->stream)); return 0; }
void* lkb_stream(lkb_ctx_t c) { return (void*)c->stream; }
int lkb_set_seed(lkb_ctx_t c, uint64_t seed) { c->seed = seed; c->seed_calls = 0; return 0; }
int lkb_set_graphs(lkb_ctx_t c, int enable) { c->graphs = enable != 0; return 0; }
int lkb_set_option(lkb_ctx_t c, const char* name, int value) {
    if (!c || !name) return LKB_ERR_ARG;
    if (!strcmp(name, "write_intermediate")) { c->write_intermediate = value != 0; return 0; }     // host-side only: graphs stay valid
    cudaStreamSynchronize(c->stream);
    invalidate_graphs(c, 0);          // cached step graphs were captured with the previous settings
    if (!strcmp(name, "graphs")) c->graphs = value != 0;
    else if (!strcmp(name, "fused")) c->fused = value != 0;
    else if (!strcmp(name, "fin")) c->fin = value != 0;
    else if (!strcmp(name, "pdl")) c->pdl = value != 0;
    else if (!strcmp(name, "serpentine")) c->serpentine = value != 0;
    else if (!strcmp(name, "csr_slice_kb")) c->csr_slice_kb = value;            // 0 disables the L2 blocking
    else if (!strcmp(name, "csr_block_min_kb")) c->csr_block_min_kb = value;
    else if (!strcmp(name, "fused_halo")) c->fused_halo = value != 0;
    else if (!strcmp(name, "p2p")) c->p2p_active = (value != 0) && c->p2p.world > 1;
    else { set_error("unknown option %s", name); return LKB_ERR_ARG; }
    return 0;
}
int lkb_p2p_export(lkb_ctx_t c, void* handle64) {
    if (!c || !handle64) return LKB_ERR_ARG;
    cudaSetDevice(c->dev);
    if (!c->p2p_region) {
        LKB_TRY(cuda_alloc(c->p2p_region, p2p_region_bytes()));
        LKB_CUDA(cudaMemset(c->p2p_region, 0, p2p_region_bytes()));
        LKB_TRY(cuda_alloc(c->p2p_epoch, 64));
        c->p2p.epoch = c->p2p_epoch;
        LKB_CUDA(cudaMemset(c->p2p.epoch, 0, 64));
        LKB_CUDA(cudaDeviceSynchronize());
    }
    cudaIpcMemHandle_t h;
    LKB_CUDA(cudaIpcGetMemHandle(&h, c->p2p_region));
    static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(handle64, &h, 64);
    return 0;
}
int lkb_p2p_attach(lkb_ctx_t c, const void* handles) {
    if (!c || !handles || !c->p2p_region) { set_error("p2p_attach: call lkb_p2p_export first"); return LKB_ERR_ARG; }
    if (c->world < 2 || c->world > P2P_MAXW) { set_error("p2p_attach: world size %d not supported (2..%d)", c->world, (int)P2P_MAXW); return LKB_ERR_ARG; }
    cudaSetDevice(c->dev);
    c->p2p.world = c->world; c->p2p.rank = c->rank;
    for (int r = 0; r < c->world; ++r) {
        if (r == c->rank) { c->p2p.peer[r] = (char*)c->p2p_region.get(); continue; }
        cudaIpcMemHandle_t h; memcpy(&h, (const char*)handles + 64 * (size_t)r, 64);
        cudaError_t e = cudaIpcOpenMemHandle(c->peer_map[r].out(), h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) { set_error("cudaIpcOpenMemHandle(rank %d) failed: %s", r, cudaGetErrorString(e)); cudaGetLastError(); return LKB_ERR_CUDA; }
        c->p2p.peer[r] = (char*)c->peer_map[r].get();
    }
    c->p2p_active = true;
    return 0;
}
int lkb_rank(lkb_ctx_t c) { return c->rank; }
int lkb_world(lkb_ctx_t c) { return c->world; }
int lkb_set_profile(lkb_ctx_t c, int enable) {
    c->profile = enable != 0;
    for (int i = 0; i < PC_COUNT; ++i) { c->prof_ms[i] = 0; c->prof_n[i] = 0; }
    return 0;
}
int lkb_get_profile(lkb_ctx_t c, double* ms8, int64_t* launches8) {
    LKB_TRY(prof_collect(c));
    for (int i = 0; i < PC_COUNT; ++i) { if (ms8) ms8[i] = c->prof_ms[i]; if (launches8) launches8[i] = c->prof_n[i]; }
    return 0;
}
int64_t lkb_kernel_launches(lkb_ctx_t c) { return c->launches; }
// In-kernel timeline of the reduction kernels (k_multidot, k_axpy_dot): %globaltimer at CTA start / main loop done /
// ticket, and around the last CTA's stage-2 fold and allreduce.  Debug / measurement only (profiles/ktime_probe.py).
int lkb_debug_ktime(lkb_ctx_t c, int enable) {
    if (!c) return LKB_ERR_ARG;
    cudaSetDevice(c->dev);
    cudaStreamSynchronize(c->stream);
    invalidate_graphs(c, 0);
    if (enable) {
        if (!c->ktime) LKB_TRY(cuda_alloc(c->ktime, KT_WORDS * sizeof(unsigned long long)));
        c->p2p.dbg = c->ktime;
        LKB_CUDA(cudaMemset(c->p2p.dbg, 0, KT_WORDS * sizeof(unsigned long long)));
    } else {
        c->ktime.reset(); c->p2p.dbg = nullptr;
    }
    return 0;
}
int lkb_debug_ktime_read(lkb_ctx_t c, uint64_t* out, int nwords) {
    if (!c || !out || !c->p2p.dbg || nwords < 0 || nwords > KT_WORDS) { set_error("ktime_read: not enabled / bad size"); return LKB_ERR_ARG; }
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    LKB_CUDA(cudaMemcpy(out, c->p2p.dbg, (size_t)nwords * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return 0;
}

// ---- vectors --------------------------------------------------------------------------------
int lkb_vec_create(lkb_ctx_t c, int kind, int64_t n_local, int64_t n_global, int64_t row0, lkb_vec_t* v) {
    if (!c || !v || kind < 0 || kind > 3 || n_local < 0) return LKB_ERR_ARG;
    cudaSetDevice(c->dev);
    lkb_vec_s* h = new lkb_vec_s{c, kind, n_local, n_global, row0, nullptr, true};
    size_t bytes = std::max((size_t)n_local * kind_size(kind), (size_t)16);
    if (dev_alloc(c, &h->d, bytes) != 0) { delete h; return LKB_ERR_ALLOC; }
    cudaMemsetAsync(h->d, 0, bytes, c->stream);
    *v = h;
    return 0;
}
int lkb_vec_wrap(lkb_ctx_t c, int kind, int64_t n_local, int64_t n_global, int64_t row0, void* devptr, lkb_vec_t* v) {
    if (!c || !v || !devptr || ((uintptr_t)devptr & 15)) { set_error("lkb_vec_wrap: pointer must be 16-byte aligned"); return LKB_ERR_ARG; }
    *v = new lkb_vec_s{c, kind, n_local, n_global, row0, devptr, false};
    return 0;
}
int lkb_vec_clone(lkb_vec_t src, lkb_vec_t* dst) {
    if (!src || !dst) return LKB_ERR_ARG;
    LKB_TRY(lkb_vec_create(src->ctx, src->kind, src->n, src->n_global, src->row0, dst));
    LKB_CUDA(cudaMemcpyAsync((*dst)->d, src->d, (size_t)src->n * kind_size(src->kind), cudaMemcpyDeviceToDevice, src->ctx->stream));
    return 0;
}
int lkb_vec_destroy(lkb_vec_t v) {
    if (!v) return LKB_ERR_ARG;
    if (v->owns && v->d) dev_free(v->ctx, v->d);
    delete v;
    return 0;
}
int lkb_vec_zero(lkb_vec_t v) {
    LKB_CUDA(cudaMemsetAsync(v->d, 0, (size_t)v->n * kind_size(v->kind), v->ctx->stream));
    return 0;
}
int lkb_vec_fill_random(lkb_vec_t v, int dist, uint64_t seed) {
    prof_launch(v->ctx, PC_OTHER, 1, [&] { launch_fill(v->kind, v->ctx->stream, v->d, v->n, v->row0, dist, seed, v->ctx->sms); });
    return check_launch(v->ctx, "fill");
}
int lkb_vec_rand(lkb_vec_t v, int32_t ifnorm) {
    LKB_TRY(lkb_vec_fill_random(v, LKB_DIST_NORMAL, next_seed(v->ctx)));
    if (ifnorm) {
        double nrm = 0;
        LKB_TRY(vec_norm_sync(v->ctx, v->kind, v->d, v->n, &nrm));
        prof_launch(v->ctx, PC_OTHER, 1, [&] { launch_scal(v->kind, v->ctx->stream, Scalar{1.0 / nrm, 0.0}, v->d, v->n, v->ctx->sms); });
        return check_launch(v->ctx, "scal");
    }
    return 0;
}
int lkb_vec_scal(lkb_vec_t v, const void* alpha) {
    prof_launch(v->ctx, PC_OTHER, 1, [&] { launch_scal(v->kind, v->ctx->stream, to_scalar(load_kind(v->kind, alpha, 0)), v->d, v->n, v->ctx->sms); });
    return check_launch(v->ctx, "scal");
}
int lkb_vec_axpby(const void* alpha, lkb_vec_t x, const void* beta, lkb_vec_t self) {
    if (!x || !self || x->n != self->n || x->kind != self->kind) { set_error("axpby: size/kind mismatch"); return LKB_ERR_ARG; }
    prof_launch(self->ctx, PC_OTHER, 1, [&] {
        launch_axpby(self->kind, self->ctx->stream, to_scalar(load_kind(self->kind, alpha, 0)), x->d, to_scalar(load_kind(self->kind, beta, 0)),
                     self->d, self->n, self->ctx->sms);
    });
    return check_launch(self->ctx, "axpby");
}
int lkb_vec_dot(lkb_vec_t self, lkb_vec_t vec, void* out) {
    if (!self || !vec || self->n != vec->n || self->kind != vec->kind) { set_error("dot: size/kind mismatch"); return LKB_ERR_ARG; }
    Scalar s;
    LKB_TRY(vec_dot_sync(self->ctx, self->kind, self->d, vec->d, self->n, &s));
    store_kind(self->kind, out, 0, cd(s.re, s.im));
    return 0;
}
int lkb_vec_norm(lkb_vec_t v, double* out) { return vec_norm_sync(v->ctx, v->kind, v->d, v->n, out); }
int64_t lkb_vec_size(lkb_vec_t v) { return v->n_global; }
int64_t lkb_vec_local_size(lkb_vec_t v) { return v->n; }
void* lkb_vec_ptr(lkb_vec_t v) { return v->d; }
int lkb_vec_put(lkb_vec_t v, const void* host) {
    LKB_CUDA(cudaMemcpyAsync(v->d, host, (size_t)v->n * kind_size(v->kind), cudaMemcpyHostToDevice, v->ctx->stream));
    LKB_CUDA(cudaStreamSynchronize(v->ctx->stream));
    return 0;
}
int lkb_vec_get(lkb_vec_t v, void* host) {
    LKB_CUDA(cudaMemcpyAsync(host, v->d, (size_t)v->n * kind_size(v->kind), cudaMemcpyDeviceToHost, v->ctx->stream));
    LKB_CUDA(cudaStreamSynchronize(v->ctx->stream));
    return 0;
}

// ---- basis ----------------------------------------------------------------------------------
int lkb_basis_create(lkb_ctx_t c, int kind, int64_t n_local, int64_t n_global, int64_t row0, int ncols, lkb_basis_t* b) {
    if (!c || !b || kind < 0 || kind > 3 || n_local < 0 || ncols < 1) return LKB_ERR_ARG;
    cudaSetDevice(c->dev);
    // columns padded to 128 B so every column starts on a full cache line / 16-byte pack boundary
    const int64_t epl = 128 / (int64_t)kind_size(kind);
    const int64_t ld = ((std::max<int64_t>(n_local, 1) + epl - 1) / epl) * epl;
    lkb_basis_s* h = new lkb_basis_s{c, kind, n_local, n_global, row0, ld, ncols, nullptr, next_uid()};
    const size_t bytes = (size_t)ld * (size_t)ncols * kind_size(kind);
    if (dev_alloc(c, &h->d, bytes) != 0) { delete h; return LKB_ERR_ALLOC; }
    cudaMemsetAsync(h->d, 0, bytes, c->stream);
    *b = h;
    return 0;
}
int lkb_basis_destroy(lkb_basis_t b) {
    if (!b) return LKB_ERR_ARG;
    invalidate_graphs(b->ctx, b->uid);
    if (b->owns) dev_free(b->ctx, b->d);
    delete b;
    return 0;
}
int lkb_basis_col(lkb_basis_t b, int i0, lkb_vec_t* view) {
    if (!b || i0 < 0 || i0 >= b->ncols) { set_error("basis_col: column %d out of range", i0); return LKB_ERR_ARG; }
    *view = new lkb_vec_s{b->ctx, b->kind, b->n, b->n_global, b->row0, col_ptr(b, i0), false};
    return 0;
}
// Non-owning view of columns [col0, col0 + ncols) of a basis: what a Fortran array section X(k1:k2) of device
// vectors maps to.  The view's identity is a fixed function of (parent, col0, ncols), so step graphs captured
// through a view are found again when the same section is passed the next time.
int lkb_basis_view(lkb_basis_t b, int col0, int ncols, lkb_basis_t* view) {
    if (!b || !view || col0 < 0 || ncols < 1 || col0 + ncols > b->ncols) { set_error("basis_view: columns [%d, %d) out of range", col0, col0 + ncols); return LKB_ERR_ARG; }
    lkb_basis_s* h = new lkb_basis_s{b->ctx, b->kind, b->n, b->n_global, b->row0, b->ld, ncols, col_ptr(b, col0),
                                     (b->uid * 1000003ULL + (uint64_t)col0 * 4099ULL + (uint64_t)ncols) | (1ULL << 62)};
    h->owns = false;
    *view = h;
    return 0;
}
// axpby_basis (AbstractVectors.fypp:697-709): Y(:, ycol0 + q) = alpha X(:, xcol0 + q) + beta Y(:, ycol0 + q); beta == 0 = copy
int lkb_basis_axpby(const void* alpha, lkb_basis_t X, int xcol0, const void* beta, lkb_basis_t Y, int ycol0, int ncols) {
    if (!X || !Y || !alpha || !beta || xcol0 < 0 || ycol0 < 0 || ncols < 0 || xcol0 + ncols > X->ncols || ycol0 + ncols > Y->ncols ||
        X->n != Y->n || X->kind != Y->kind) { set_error("basis_axpby: bad arguments"); return LKB_ERR_ARG; }
    lkb_ctx_s* c = Y->ctx;
    const Scalar a = to_scalar(load_kind(Y->kind, alpha, 0)), bb = to_scalar(load_kind(Y->kind, beta, 0));
    for (int q = 0; q < ncols; ++q)
        prof_launch(c, PC_OTHER, 1, [&] { launch_axpby(Y->kind, c->stream, a, col_ptr(X, xcol0 + q), bb, col_ptr(Y, ycol0 + q), Y->n, c->sms); });
    return check_launch(c, "basis_axpby");
}
// rand_basis (AbstractVectors.fypp:725-730)
int lkb_basis_rand(lkb_basis_t b, int col0, int ncols, int32_t ifnorm) {
    if (!b || col0 < 0 || ncols < 0 || col0 + ncols > b->ncols) { set_error("basis_rand: bad arguments"); return LKB_ERR_ARG; }
    lkb_ctx_s* c = b->ctx;
    for (int q = 0; q < ncols; ++q) {
        void* w = col_ptr(b, col0 + q);
        prof_launch(c, PC_OTHER, 1, [&] { launch_fill(b->kind, c->stream, w, b->n, b->row0, LKB_DIST_NORMAL, next_seed(c), c->sms); });
        if (ifnorm) {
            double nrm = 0;
            LKB_TRY(vec_norm_sync(c, b->kind, w, b->n, &nrm));
            prof_launch(c, PC_OTHER, 1, [&] { launch_scal(b->kind, c->stream, Scalar{1.0 / nrm, 0.0}, w, b->n, c->sms); });
        }
    }
    return check_launch(c, "basis_rand");
}
int lkb_basis_zero(lkb_basis_t b, int col0, int ncols) {
    if (col0 < 0 || col0 + ncols > b->ncols) return LKB_ERR_ARG;
    LKB_CUDA(cudaMemsetAsync(col_ptr(b, col0), 0, (size_t)b->ld * ncols * kind_size(b->kind), b->ctx->stream));
    return 0;
}
int lkb_basis_put(lkb_basis_t b, int col0, int ncols, const void* host, int64_t ldhost) {
    if (col0 < 0 || col0 + ncols > b->ncols) return LKB_ERR_ARG;
    const size_t es = kind_size(b->kind);
    LKB_CUDA(cudaMemcpy2DAsync(col_ptr(b, col0), (size_t)b->ld * es, host, (size_t)ldhost * es, (size_t)b->n * es, ncols,
                               cudaMemcpyHostToDevice, b->ctx->stream));
    LKB_CUDA(cudaStreamSynchronize(b->ctx->stream));
    return 0;
}
int lkb_basis_get(lkb_basis_t b, int col0, int ncols, void* host, int64_t ldhost) {
    if (col0 < 0 || col0 + ncols > b->ncols) return LKB_ERR_ARG;
    const size_t es = kind_size(b->kind);
    LKB_CUDA(cudaMemcpy2DAsync(host, (size_t)ldhost * es, col_ptr(b, col0), (size_t)b->ld * es, (size_t)b->n * es, ncols,
                               cudaMemcpyDeviceToHost, b->ctx->stream));
    LKB_CUDA(cudaStreamSynchronize(b->ctx->stream));
    return 0;
}
int lkb_basis_ncols(lkb_basis_t b) { return b->ncols; }
int64_t lkb_basis_ld(lkb_basis_t b) { return b->ld; }

// ---- operators ------------------------------------------------------------------------------
static int stencil_create(lkb_ctx_t c, int kind, int dim, int64_t nx, int64_t ny, int64_t nz, const void* coef,
                          int64_t slow0, int64_t nslow_local, lkb_op_t* A) {
    if (!c || !A || !coef || nx < 1 || ny < 1 || nz < 1) return LKB_ERR_ARG;
    const int64_t nslow = dim == 2 ? ny : nz;
    if (slow0 < 0 || nslow_local < 1 || slow0 + nslow_local > nslow) { set_error("stencil: bad slab [%lld,+%lld) of %lld", (long long)slow0, (long long)nslow_local, (long long)nslow); return LKB_ERR_ARG; }
    cudaSetDevice(c->dev);
    OpOwner op(new lkb_op_s());
    op->ctx = c; op->type = OP_STENCIL; op->kind = kind; op->uid = next_uid();
    op->st.dim = dim; op->st.nx = nx;
    op->st.ny = dim == 2 ? nslow_local : ny;
    op->st.nz = dim == 2 ? 1 : nslow_local;
    op->slow0 = slow0; op->nslow_global = nslow;
    const int ncoef = dim == 2 ? 5 : 7;
    const size_t es = kind_size(kind);
    for (int q = 0; q < 7; ++q) op->st.coef[q] = q < ncoef ? to_scalar(load_kind(kind, coef, q)) : Scalar{0, 0};
    op->m = op->n = nx * op->st.ny * op->st.nz;
    op->halo_elems = dim == 2 ? nx : nx * ny;
    op->st.halo_lo = op->st.halo_hi = nullptr;
    if (c->world > 1) {
        // (NCCL-halo fallback buffers; a failure here is local, but nothing collective has been issued yet)
        LKB_TRY(cuda_alloc(op->halo_lo, op->halo_elems * es));
        LKB_TRY(cuda_alloc(op->halo_hi, op->halo_elems * es));
        if (slow0 > 0) op->st.halo_lo = op->halo_lo;
        if (slow0 + nslow_local < nslow) op->st.halo_hi = op->halo_hi;
        if (c->p2p_active) {
            // P2P halo exchange: a double-buffered halo region per rank, mapped into both neighbours with
            // CUDA IPC (handles all-gathered over the context's NCCL communicator: creation is collective)
            NcclApi* api = nccl_api();
            const size_t side = (((size_t)op->halo_elems * es) + 255) & ~(size_t)255;
            const size_t region = 256 + 4 * side;
            CudaPtr<void> reg, hbuf; CudaPtr<unsigned> ctr; IpcMap lo_map, hi_map;     // installed in op only when every rank succeeded
            bool ok = api && cuda_alloc(reg, region) == 0 && cudaMemset(reg, 0, region) == cudaSuccess &&
                      cuda_alloc(hbuf, 64 * (size_t)(c->world + 1)) == 0 &&
                      cuda_alloc(ctr, 128) == 0 && cudaMemset(ctr, 0, 128) == cudaSuccess;
            std::vector<char> all(64 * (size_t)c->world);
            if (ok) {
                cudaIpcMemHandle_t hnd;
                ok = cudaIpcGetMemHandle(&hnd, reg) == cudaSuccess &&
                     cudaMemcpy((char*)hbuf.get() + 64 * (size_t)c->world, &hnd, 64, cudaMemcpyHostToDevice) == cudaSuccess;
            }
            // the all-gather is issued unconditionally so that the ranks stay in step even if one failed locally
            int okflag = ok ? 1 : 0;
            if (api && hbuf) {
                if (api->AllGather((char*)hbuf.get() + 64 * (size_t)c->world, hbuf, 64, /*ncclInt8*/ 0, c->comm, c->stream) != 0) okflag = 0;
                if (cudaMemcpyAsync(all.data(), hbuf, all.size(), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) okflag = 0;
                if (cudaStreamSynchronize(c->stream) != cudaSuccess) okflag = 0;
            } else okflag = 0;
            const bool has_lo = slow0 > 0, has_hi = slow0 + nslow_local < nslow;
            if (okflag && has_lo) {
                cudaIpcMemHandle_t hnd; memcpy(&hnd, &all[64 * (size_t)(c->rank - 1)], 64);
                if (cudaIpcOpenMemHandle(lo_map.out(), hnd, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { okflag = 0; cudaGetLastError(); }
            }
            if (okflag && has_hi) {
                cudaIpcMemHandle_t hnd; memcpy(&hnd, &all[64 * (size_t)(c->rank + 1)], 64);
                if (cudaIpcOpenMemHandle(hi_map.out(), hnd, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { okflag = 0; cudaGetLastError(); }
            }
            hbuf.reset();
            // every rank must take the same path: agree through one more (tiny) all-reduce-like exchange
            if (ensure_ws(c, 2) != 0) okflag = 0;     // (never return before the agreement step: the ranks would desynchronise)
            {
                double v = okflag ? 0.0 : 1.0;
                cudaMemcpyAsync(c->tmpw, &v, sizeof(double), cudaMemcpyHostToDevice, c->stream);
                if (api) api->AllReduce(c->tmpw, c->tmpw, 1, 8, 0, c->comm, c->stream);
                cudaMemcpyAsync(&v, c->tmpw, sizeof(double), cudaMemcpyDeviceToHost, c->stream);
                cudaStreamSynchronize(c->stream);
                if (v != 0.0) okflag = 0;
            }
            if (okflag) {
                op->hp.my_region = (char*)reg.get(); op->hp.lo_region = (char*)lo_map.get(); op->hp.hi_region = (char*)hi_map.get();
                op->hp.epoch = ctr; op->hp.ticket = ctr.get() + 16; op->hp.he = op->halo_elems;
                op->hp.data_off = 256; op->hp.side_bytes = side;
                op->hp_active = true;
                if (has_lo) op->st.halo_lo = (char*)reg.get() + 256;              // parity 0, side 0
                if (has_hi) op->st.halo_hi = (char*)reg.get() + 256 + side;       // parity 0, side 1
                op->st.halo_epoch = ctr;
                op->st.halo_parity_stride = (int64_t)(2 * side / es);
                op->st.flag_lo = (const unsigned*)reg.get();                      // "lower neighbour pushed epoch e"
                op->st.flag_hi = (const unsigned*)((char*)reg.get() + 128);       // "upper neighbour pushed epoch e"
                op->hp_region = std::move(reg); op->hp_ctr = std::move(ctr); op->hp_lo_map = std::move(lo_map); op->hp_hi_map = std::move(hi_map);
            }
        }
    }
    const int64_t gy = ((op->st.ny + 7) / 8) * op->st.nz * (nx / 128 + 1);     // upper bound on the 1-D grid of the stencil kernels
    if (gy > 2147483647LL) { set_error("stencil: grid too large for this kernel (%lld CTAs)", (long long)gy); return LKB_ERR_ARG; }
    *A = op.release();
    return 0;
}
int lkb_op_stencil5_create(lkb_ctx_t c, int kind, int64_t nx, int64_t ny, const void* coef5, int64_t slow0,
                           int64_t nslow_local, lkb_op_t* A) {
    return stencil_create(c, kind, 2, nx, ny, 1, coef5, slow0, nslow_local, A);
}
int lkb_op_stencil7_create(lkb_ctx_t c, int kind, int64_t nx, int64_t ny, int64_t nz, const void* coef7, int64_t slow0,
                           int64_t nslow_local, lkb_op_t* A) {
    return stencil_create(c, kind, 3, nx, ny, nz, coef7, slow0, nslow_local, A);
}

// Row-sharded CSR (SURVEY 8e): this rank owns rows [row0, row0+m_local) of the m_global x n_global matrix with
// GLOBAL column indices; input vectors of matvec are sharded over the column space as [col0, col0+n_local).
//   matvec : all ranks' slabs of x are gathered into a full-length buffer (grouped ncclBroadcast, ragged slabs
//            allowed), then the local SpMV runs;   rmatvec: the local A_loc^H u_loc contributes to all n_global
//            entries, each slab is summed onto its owner (grouped ncclReduce).  Creation is collective.
// slab bookkeeping + gather / reduce buffers of a row-sharded CSR operator whose local arrays are already in place
static int csr_dist_finish(lkb_ctx_t c, lkb_op_s* op, int kind, int64_t n_global, int64_t row0, int64_t m_local, int64_t col0, int64_t n_local) {
    const size_t es = kind_size(kind);
    // every rank's slab of the column and row spaces
    const int W = c->world;
    op->col_off.assign(W, 0); op->col_cnt.assign(W, 0); op->row_off.assign(W, 0); op->row_cnt.assign(W, 0);
    if (W == 1) {
        op->col_off[0] = col0; op->col_cnt[0] = n_local; op->row_off[0] = row0; op->row_cnt[0] = m_local;
    } else {
        NcclApi* api = nccl_api();
        if (!api) return LKB_ERR_NCCL;
        const int64_t mine[4] = {col0, n_local, row0, m_local};
        std::vector<int64_t> all(4 * (size_t)W);
        CudaPtr<char> dbuf;
        LKB_TRY(cuda_alloc(dbuf, 32 * (size_t)(W + 1)));
        bool ok = cudaMemcpy(dbuf.get() + 32 * (size_t)W, mine, 32, cudaMemcpyHostToDevice) == cudaSuccess &&
                  api->AllGather(dbuf.get() + 32 * (size_t)W, dbuf, 32, /*ncclInt8*/ 0, c->comm, c->stream) == 0 &&
                  cudaMemcpyAsync(all.data(), dbuf, 32 * (size_t)W, cudaMemcpyDeviceToHost, c->stream) == cudaSuccess &&
                  cudaStreamSynchronize(c->stream) == cudaSuccess;
        if (!ok) { set_error("csr_create_dist: slab exchange failed"); return LKB_ERR_NCCL; }
        for (int q = 0; q < W; ++q) { op->col_off[q] = all[4 * q]; op->col_cnt[q] = all[4 * q + 1]; op->row_off[q] = all[4 * q + 2]; op->row_cnt[q] = all[4 * q + 3]; }
    }
    LKB_TRY(cuda_alloc(op->x_full, std::max<size_t>((size_t)n_global * es, 16)));
    LKB_TRY(cuda_alloc(op->y_full, std::max<size_t>((size_t)n_global * es, 16)));
    return cuda_alloc(op->y_red, std::max<size_t>((size_t)n_local * es, 16));
}
int lkb_op_csr_create_dist(lkb_ctx_t c, int kind, int64_t m_global, int64_t n_global, int64_t row0, int64_t m_local,
                           int64_t col0, int64_t n_local, const int64_t* rowptr_local, const int32_t* col_global,
                           const void* val, lkb_op_t* A) {
    if (!c || !A || !rowptr_local || m_local < 0 || n_local < 0 || m_global < 1 || n_global < 1) return LKB_ERR_ARG;
    cudaSetDevice(c->dev);
    OpOwner op(new lkb_op_s());
    op->ctx = c; op->type = OP_CSR; op->kind = kind; op->m = m_local; op->n = n_local; op->uid = next_uid();
    op->dist = true; op->m_global = m_global; op->n_global = n_global;
    LKB_TRY(csr_dist_finish(c, op, kind, n_global, row0, m_local, col0, n_local));
    LKB_TRY(csr_build(c, op, kind, m_local, n_global, rowptr_local, col_global, val));
    *A = op.release();
    return 0;
}
// The same from local CSR arrays that already live on this GPU (e.g. lkb_csr_random_device); adopt as in lkb_op_csr_create_device.
int lkb_op_csr_create_dist_device(lkb_ctx_t c, int kind, int64_t m_global, int64_t n_global, int64_t row0, int64_t m_local,
                                  int64_t col0, int64_t n_local, int64_t* rowptr_dev, int32_t* col_dev, void* val_dev,
                                  int32_t adopt, lkb_op_t* A) {
    if (!c || !A || !rowptr_dev || !col_dev || !val_dev || m_local < 1 || n_local < 0 || m_global < 1 || n_global < 1 || kind < 0 || kind > 3)
        { set_error("csr_create_dist_device: bad arguments"); return LKB_ERR_ARG; }
    if (!adopt) { set_error("csr_create_dist_device: only adopt != 0 is supported"); return LKB_ERR_ARG; }
    cudaSetDevice(c->dev);
    OpOwner op(new lkb_op_s());
    op->ctx = c; op->type = OP_CSR; op->kind = kind; op->m = m_local; op->n = n_local; op->uid = next_uid();
    op->dist = true; op->m_global = m_global; op->n_global = n_global;
    // the slab exchange comes first: once csr_finish_device has succeeded, the adopted arrays may have been released
    LKB_TRY(csr_dist_finish(c, op, kind, n_global, row0, m_local, col0, n_local));
    op->rowptr.reset(rowptr_dev); op->col.reset(col_dev); op->val.reset(val_dev);
    if (int r = csr_finish_device(c, op, kind, m_local, n_global)) {
        op->rowptr.release(); op->col.release(); op->val.release();      // the caller keeps ownership on failure
        return r;
    }
    *A = op.release();
    return 0;
}
int lkb_op_dense_create(lkb_ctx_t c, int kind, int64_t m, int64_t n, const void* a, lkb_op_t* A) {
    if (!c || !A || !a || m < 1 || n < 1) return LKB_ERR_ARG;
    if (c->world > 1) { set_error("dense operators are single-rank (plumbing config only)"); return LKB_ERR_ARG; }
    cudaSetDevice(c->dev);
    OpOwner op(new lkb_op_s());
    op->ctx = c; op->type = OP_DENSE; op->kind = kind; op->m = m; op->n = n; op->uid = next_uid();
    LKB_TRY(cuda_alloc(op->a, (size_t)m * n * kind_size(kind)));
    LKB_CUDA(cudaMemcpy(op->a, a, (size_t)m * n * kind_size(kind), cudaMemcpyHostToDevice));
    *A = op.release();
    return 0;
}
int lkb_op_callback_create(lkb_ctx_t c, int kind, int64_t m_local, int64_t n_local, lkb_matvec_fn fn, void* user,
                           int32_t capturable, lkb_op_t* A) {
    if (!c || !A || !fn) return LKB_ERR_ARG;
    lkb_op_s* op = new lkb_op_s();
    op->ctx = c; op->type = OP_CALLBACK; op->kind = kind; op->m = m_local; op->n = n_local; op->uid = next_uid();
    op->fn = fn; op->user = user; op->capturable = capturable != 0;
    *A = op;
    return 0;
}
// Diagonal operator M = diag(d), e.g. the inverse mass matrix of a spectral-element code.  Row-local, so it has
// the layout of d and needs no communication at N > 1.  Its values are copied: d may be released afterwards.
static int diag_from_device(lkb_ctx_t c, int kind, int64_t n, int64_t row0, int64_t n_global, OpOwner& op) {
    cudaSetDevice(c->dev);
    op.reset(new lkb_op_s());
    op->ctx = c; op->type = OP_DIAG; op->kind = kind; op->m = op->n = n; op->uid = next_uid();
    op->diag_row0 = row0; op->diag_n_global = n_global;
    return cuda_alloc(op->diag, std::max<size_t>((size_t)n * kind_size(kind), 16));
}
int lkb_op_diag_create(lkb_vec_t d, lkb_op_t* M) {
    if (!d || !M) { set_error("diag_create: null argument"); return LKB_ERR_ARG; }
    lkb_ctx_s* c = d->ctx;
    OpOwner op;
    LKB_TRY(diag_from_device(c, d->kind, d->n, d->row0, d->n_global, op));
    if (cudaMemcpyAsync(op->diag, d->d, (size_t)d->n * kind_size(d->kind), cudaMemcpyDeviceToDevice, c->stream) != cudaSuccess ||
        cudaStreamSynchronize(c->stream) != cudaSuccess) {
        set_error("diag_create: copy of d failed: %s", cudaGetErrorString(cudaGetLastError()));
        return LKB_ERR_CUDA;
    }
    *M = op.release();
    return 0;
}
// Jacobi preconditioner M = diag(A)^-1, found and inverted on the device (k_jacobi).  Not collective: a rank whose slab
// holds a zero or non-finite diagonal entry reports it, with the first such global row.
int lkb_op_jacobi_create(lkb_op_t A, lkb_op_t* M) {
    if (!A || !M) { set_error("jacobi_create: null argument"); return LKB_ERR_ARG; }
    lkb_ctx_s* c = A->ctx;
    if (A->type == OP_CALLBACK) { set_error("jacobi_create: a callback operator has no diagonal the library can read"); return LKB_ERR_ARG; }
    if (A->m != A->n) { set_error("jacobi_create: A is not square (%lld x %lld local rows / columns)", (long long)A->m, (long long)A->n); return LKB_ERR_ARG; }
    JacobiSrc src;
    src.rows = A->m;
    int64_t n_global = A->m;
    if (A->type == OP_STENCIL) {
        const int64_t plane = A->st.dim == 2 ? A->st.nx : A->st.nx * A->st.ny;
        src.mode = JAC_STENCIL; src.c0 = A->st.coef[0];
        src.row0 = A->slow0 * plane; n_global = A->nslow_global * plane;
    } else if (A->type == OP_CSR) {
        if (A->dist) {
            const int r = c->rank;
            if (A->row_off[r] != A->col_off[r] || A->row_cnt[r] != A->col_cnt[r] || A->m_global != A->n_global) {
                set_error("jacobi_create: row-sharded CSR whose row slab [%lld,+%lld) differs from its column slab [%lld,+%lld) "
                          "on rank %d (the diagonal is defined only when they agree)", (long long)A->row_off[r], (long long)A->row_cnt[r],
                          (long long)A->col_off[r], (long long)A->col_cnt[r], r);
                return LKB_ERR_ARG;
            }
            src.row0 = src.col0 = A->row_off[r]; n_global = A->n_global;
        }
        if (A->blk.nb > 0) { src.mode = JAC_CSR_BLOCKED; src.blk = A->blk; }
        else { src.mode = JAC_CSR; src.rowptr = A->rowptr; src.col = A->col; src.val = A->val; }
    } else if (A->type == OP_DENSE) {
        src.mode = JAC_DENSE; src.a = A->a;
    } else if (A->type == OP_DIAG) {
        src.mode = JAC_DIAG; src.a = A->diag; src.row0 = A->diag_row0; n_global = A->diag_n_global;
    } else {
        set_error("jacobi_create: unsupported operator type %d", A->type); return LKB_ERR_ARG;
    }
    OpOwner op;
    LKB_TRY(diag_from_device(c, A->kind, A->m, src.row0, n_global, op));
    CudaPtr<unsigned long long> bad; unsigned long long hbad = 0;
    LKB_TRY(cuda_alloc(bad, sizeof(unsigned long long)));
    LKB_CUDA(cudaMemsetAsync(bad, 0xff, sizeof(unsigned long long), c->stream));
    launch_jacobi(A->kind, c->stream, src, op->diag, bad, c->sms);
    LKB_TRY(check_launch(c, "jacobi"));
    LKB_CUDA(cudaMemcpyAsync(&hbad, bad, sizeof(hbad), cudaMemcpyDeviceToHost, c->stream));
    LKB_CUDA(cudaStreamSynchronize(c->stream));
    if (hbad != ~0ULL) {
        set_error("jacobi_create: the diagonal entry of global row %llu is zero or not finite", hbad);
        return LKB_ERR_ARG;
    }
    *M = op.release();
    return 0;
}
int lkb_op_destroy(lkb_op_t A) {
    if (!A) return LKB_ERR_ARG;
    cudaStreamSynchronize(A->ctx->stream);
    invalidate_graphs(A->ctx, A->uid);
    delete A;
    return 0;
}
int lkb_op_counters(lkb_op_t A, int64_t* n_matvec, int64_t* n_rmatvec) {
    if (n_matvec) *n_matvec = A->n_matvec;
    if (n_rmatvec) *n_rmatvec = A->n_rmatvec;
    return 0;
}
int lkb_op_reset_counters(lkb_op_t A) { A->n_matvec = A->n_rmatvec = 0; return 0; }

}  // extern "C"

namespace lkb {
const HaloP2P* op_halo_desc(const lkb_op_s* A, int j) {
    const lkb_ctx_s* c = A->ctx;
    return (A->type == OP_STENCIL && c->world > 1 && A->hp_active && c->fused_halo && fin_usable(c, j)) ? &A->hp : nullptr;
}
int op_apply_enqueue(lkb_op_s* A, const void* x, void* y, bool trans, const int* flags, bool halo_prepushed) {
    lkb_ctx_s* c = A->ctx;
    const size_t es = kind_size(A->kind);
    int nl = 1;
    prof_begin(c, PC_MATVEC);
    if (A->type == OP_STENCIL) {
        if (c->world > 1 && A->hp_active) {
            // halo exchange over NVLink peer memory: pushed by the kernel that finished x, or by k_halo_push
            // (copy + synchronisation in one kernel)
            if (!halo_prepushed) { launch_halo_push(A->kind, c->stream, A->hp, x, A->m, flags); nl = 2; }
        } else if (c->world > 1) {
            // halo exchange over NCCL send/recv: my first row/plane -> rank-1's halo_hi, my last -> rank+1's halo_lo
            NcclApi* api = nccl_api();
            if (!api) return LKB_ERR_NCCL;
            const int64_t he = A->halo_elems;
            const int64_t nloc = A->m;
            const size_t cnt = (size_t)he * (kind_cplx(A->kind) ? 2 : 1);
            const int dt = (A->kind == KS || A->kind == KC) ? 7 : 8;   // ncclFloat32 / ncclFloat64
            const bool has_lo = A->st.halo_lo != nullptr, has_hi = A->st.halo_hi != nullptr;
            LKB_NCCL(api->GroupStart());
            if (has_lo) {
                LKB_NCCL(api->Send(x, cnt, dt, c->rank - 1, c->comm, c->stream));
                LKB_NCCL(api->Recv(A->halo_lo, cnt, dt, c->rank - 1, c->comm, c->stream));
            }
            if (has_hi) {
                LKB_NCCL(api->Send((const char*)x + (size_t)(nloc - he) * es, cnt, dt, c->rank + 1, c->comm, c->stream));
                LKB_NCCL(api->Recv(A->halo_hi, cnt, dt, c->rank + 1, c->comm, c->stream));
            }
            LKB_NCCL(api->GroupEnd());
            pdl_rearm();
        }
        launch_stencil(A->kind, c->stream, A->st, x, y, trans, flags, c->sms);
    } else if (A->type == OP_CSR && A->dist) {
        const int dt = (A->kind == KS || A->kind == KC) ? 7 : 8;            // ncclFloat32 / ncclFloat64
        const size_t per = kind_cplx(A->kind) ? 2 : 1;
        NcclApi* api = c->world > 1 ? nccl_api() : nullptr;
        if (c->world > 1 && !api) return LKB_ERR_NCCL;
        if (!trans) {
            // gather every rank's slab of x at its true offset (ragged slabs), then the local SpMV
            if (c->world > 1) {
                LKB_NCCL(api->GroupStart());
                for (int q = 0; q < c->world; ++q) {
                    void* dst = (char*)A->x_full.get() + (size_t)A->col_off[q] * es;
                    LKB_NCCL(api->Broadcast(q == c->rank ? x : dst, dst, (size_t)A->col_cnt[q] * per, dt, q, c->comm, c->stream));
                }
                LKB_NCCL(api->GroupEnd());
            } else {
                LKB_CUDA(cudaMemcpyAsync((char*)A->x_full.get() + (size_t)A->col_off[0] * es, x, (size_t)A->n * es, cudaMemcpyDeviceToDevice, c->stream));
            }
            if (A->blk.nb > 0) { launch_csr_blocked(A->kind, c->stream, A->blk, A->x_full, y, false, flags, c->sms); nl = A->blk.nb; }
            else launch_csr(A->kind, c->stream, A->m, A->rowptr, A->col, A->val, A->x_full, y, false, flags, c->sms | (A->lpr << 16));
        } else {
            // local A_loc^H u_loc over the whole column space, then every slab is summed onto its owner
            launch_csr(A->kind, c->stream, A->n_global, A->t_rowptr, A->t_col, A->t_val, x, A->y_full, true, flags, c->sms | (A->t_lpr << 16));
            if (c->world > 1) {
                LKB_NCCL(api->GroupStart());
                // reduce into a scratch slab, then a flags-gated copy: after a device-side stop the reference leaves the
                // later basis columns untouched, so stale reductions must not land in y
                for (int q = 0; q < c->world; ++q)
                    LKB_NCCL(api->Reduce((char*)A->y_full.get() + (size_t)A->col_off[q] * es, A->y_red, (size_t)A->col_cnt[q] * per, dt, /*ncclSum*/ 0, q, c->comm, c->stream));
                LKB_NCCL(api->GroupEnd());
                launch_copy_gated(A->kind, c->stream, A->y_red, y, A->n, flags, c->sms);
                nl = 2;
            } else {
                LKB_CUDA(cudaMemcpyAsync(y, (char*)A->y_full.get() + (size_t)A->col_off[0] * es, (size_t)A->n * es, cudaMemcpyDeviceToDevice, c->stream));
            }
        }
    } else if (A->type == OP_CSR) {
        if (!trans) {
            if (A->blk.nb > 0) { launch_csr_blocked(A->kind, c->stream, A->blk, x, y, false, flags, c->sms); nl = A->blk.nb; }
            else launch_csr(A->kind, c->stream, A->m, A->rowptr, A->col, A->val, x, y, false, flags, c->sms | (A->lpr << 16));
        } else {
            if (A->t_blk.nb > 0) { launch_csr_blocked(A->kind, c->stream, A->t_blk, x, y, true, flags, c->sms); nl = A->t_blk.nb; }
            else launch_csr(A->kind, c->stream, A->n, A->t_rowptr, A->t_col, A->t_val, x, y, true, flags, c->sms | (A->t_lpr << 16));
        }
    } else if (A->type == OP_DENSE) {
        launch_dense(A->kind, c->stream, A->m, A->n, A->a, x, y, trans, flags);
    } else if (A->type == OP_DIAG) {
        launch_diag(A->kind, c->stream, A->diag, x, y, A->m, trans, flags, c->sms);      // row-local: no exchange at N > 1
    } else {
        int r = A->fn(A->user, x, y, trans ? 1 : 0, (void*)c->stream);
        if (r != 0) { set_error("user matvec callback returned %d", r); return LKB_ERR_ARG; }
        nl = 0;
    }
    // anything but our own plain kernels (NCCL gathers / reductions, device-to-device copies, a user callback) breaks
    // the programmatic-launch chain: the next PDL-aware kernel is launched normally.  The diagonal operator is one plain
    // kernel (k_diag, launched without the PDL attribute, like the stencil): a PDL-aware successor waits for its completion
    // in griddepcontrol.wait, so it keeps the chain.
    if (!(A->type == OP_STENCIL || A->type == OP_DENSE || A->type == OP_DIAG || (A->type == OP_CSR && !A->dist))) pdl_rearm();
    prof_end(c, PC_MATVEC, nl);
    return check_launch(c, "matvec");
}
}  // namespace lkb

extern "C" {
static int op_apply_api(lkb_op_t A, lkb_vec_t x, lkb_vec_t y, bool trans) {
    if (!A || !x || !y) return LKB_ERR_ARG;
    const int64_t nin = trans ? A->m : A->n, nout = trans ? A->n : A->m;
    if (x->n != nin || y->n != nout || x->kind != A->kind || y->kind != A->kind) { set_error("matvec: size/kind mismatch"); return LKB_ERR_ARG; }
    if (x->d == y->d && A->type != OP_DIAG) { set_error("matvec: vec_out must not alias vec_in"); return LKB_ERR_ARG; }   // (k_diag works in place)
    if (trans) A->n_rmatvec++; else A->n_matvec++;
    return op_apply_enqueue(A, x->d, y->d, trans, nullptr);
}
int lkb_op_matvec(lkb_op_t A, lkb_vec_t x, lkb_vec_t y) { return op_apply_api(A, x, y, false); }
int lkb_op_rmatvec(lkb_op_t A, lkb_vec_t x, lkb_vec_t y) { return op_apply_api(A, x, y, true); }
}  // extern "C"
