// C ABI of vbmf_b200 (include/vbmf_b200.h): context, resident solver state, step functions, the device-side loop.
#include "../../include/vbmf_b200.h"
#include "common.cuh"
#include "gemm.cuh"
#include "kernels.cuh"

#include <atomic>
#include <type_traits>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <unistd.h>
#include <string>
#include <vector>
#include <algorithm>
#include <thread>

namespace vb {

static thread_local char g_err[1024] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

// ------------------------------------------------------------------------------------------- NCCL (loaded at run time)
struct NcclUniqueId { char internal[128]; };
struct NcclApi {
    void* handle = nullptr;
    int (*GetUniqueId)(NcclUniqueId*) = nullptr;
    int (*CommInitRank)(void**, int, NcclUniqueId, int) = nullptr;
    int (*CommInitAll)(void**, int, const int*) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;
static int load_nccl() {
    if (g_nccl.handle) return 0;
    const char* names[] = {getenv("VBMF_B200_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    void* h = nullptr;
    for (const char* n : names) {
        if (n == nullptr || *n == 0) continue;
        h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (h) break;
    }
    if (!h) { set_error("NCCL not found (set VBMF_B200_NCCL_LIB): %s", dlerror()); return -1; }
    g_nccl.GetUniqueId = (int (*)(NcclUniqueId*))dlsym(h, "ncclGetUniqueId");
    g_nccl.CommInitRank = (int (*)(void**, int, NcclUniqueId, int))dlsym(h, "ncclCommInitRank");
    g_nccl.CommInitAll = (int (*)(void**, int, const int*))dlsym(h, "ncclCommInitAll");
    g_nccl.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(h, "ncclAllReduce");
    g_nccl.AllGather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(h, "ncclAllGather");
    g_nccl.CommDestroy = (int (*)(void*))dlsym(h, "ncclCommDestroy");
    g_nccl.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.CommDestroy) {
        set_error("NCCL library lacks a required symbol");
        return -1;
    }
    g_nccl.handle = h;
    return 0;
}
#define VB_NCCL_OK(call)                                                                        \
    do {                                                                                        \
        int r__ = (call);                                                                       \
        if (r__ != 0) {                                                                         \
            vb::set_error("%s failed: %s", #call, g_nccl.GetErrorString ? g_nccl.GetErrorString(r__) : "?"); \
            return -1;                                                                          \
        }                                                                                       \
    } while (0)

}  // namespace vb

using namespace vb;

// ------------------------------------------------------------------------------------------- context
struct vbmf_b200_ctx {
    int device = 0, rank = 0, world = 1, num_sms = 148;
    cudaStream_t st = nullptr;
    bool own_stream = false;
    void* comm = nullptr;
    // resident shard of Y (column-major L x Mloc, leading dimension ldY)
    double* Y = nullptr;
    size_t Y_cap = 0;         // bytes allocated behind Y (the buffer is reused by the next attach when it fits)
    int L_cap = 0;            // rows rowY2 / stats_part were sized for
    int L = 0, Mloc = 0, Mglob = 0, moff = 0, ldY = 0;
    double* rowY2 = nullptr;
    double* d_tr = nullptr;
    double* stats_part = nullptr;
    double trYTY = 0.0;
    CUtensorMap tmY1, tmY2;
    bool have_Y = false;
    // Large uploads travel in column chunks on a copy stream; K0 (row norms, trYTY) follows chunk by chunk on a statistics
    // stream.  Until somebody needs all of Y the main stream is free: the first dense iteration works through the chunks as
    // they arrive (enq_iteration_chunked), everything else waits for ev_stats once (ctx_wait_upload).
    cudaStream_t copy_st = nullptr, stat_st = nullptr;
    std::vector<cudaEvent_t> ev_chunk;
    std::vector<int> chunk_c0, chunk_n;
    cudaEvent_t ev_stats = nullptr;
    int chunks_pending = 0;           // > 0: chunks whose arrival the main stream has not been ordered after yet
    bool tr_pending = false;          // trYTY lives in d_tr only (not yet read back to the host)
    bool simt = false;
    bool gemm_dmma = false;   // VBMF_B200_GEMM=dmma: keep the FP64 tensor-core contractions at H <= 64 (A/B measurements)
    // int8 digit planes of Y for the INT8 contractions (gemm_int8.cu): [I8_NSL][Mloc][ldZ], exponents F[L] | E[Mloc]; built
    // on first use after every change of Y (ctx_slices)
    uint8_t* Z = nullptr;
    int* Zexp = nullptr;
    size_t Z_bytes = 0;
    int ldZ = 0;
    bool z_ready = false, z_failed = false;
    CUtensorMap tmZ1, tmZ2;
    // profiling of the two contractions
    bool profile = false;
    std::vector<cudaEvent_t> ev_k1, ev_k2, ev_ar;      // K1, K2 and (world > 1) the per-iteration all-reduce
    std::vector<std::pair<int, cudaEvent_t>> ev_seg;   // (segment tag, event at the segment's end): where an iteration's time goes
    // peer exchange (kernels.cuh, PxDev): this rank's peer-visible buffer and the peers' buffers as mapped into this device
    struct Px {
        bool ok = false, failed = false, claimed = false;
        char* local = nullptr;
        size_t cap = 0;
        char* peer[PX_MAX_WORLD] = {};
        bool ipc[PX_MAX_WORLD] = {};
        char* xchg = nullptr;             // device staging of the handle exchange
        unsigned long long epoch = 0;     // barrier epochs consumed so far (identical on every rank)
        unsigned long long* wait_ns = nullptr;   // device [3][2]: barrier wait of CTA 0 per site (profiling with segments only)
    } px;
    bool profile_segments = false;        // vbmf_b200_ctx_profile(ctx, 3): also mark the segments of every iteration (adds event records)
    // grow-only staging for the batched small-problem path (device arena + pinned host mirror, same offsets)
    char* batch_dev = nullptr;
    char* batch_host = nullptr;
    size_t batch_bytes = 0;
};

static int ctx_allreduce(vbmf_b200_ctx* c, double* buf, size_t n) {
    if (c->world <= 1 || n == 0) return 0;
    VB_NCCL_OK(g_nccl.AllReduce(buf, buf, n, /*ncclFloat64*/ 8, /*ncclSum*/ 0, c->comm, c->st));
    return 0;
}

// ------------------------------------------------------------------------------------------- peer exchange set-up
// One peer-visible buffer per rank, mapped into every other rank's device: cudaIpc handles between processes (one process per
// GPU), plain peer access inside one process (vbmf_b200_mctx_*).  The handles travel through the communicator the context
// already has; the outcome is agreed on by all ranks (one failing rank switches the exchange off everywhere, the NCCL
// all-reduce path stays).  Collective: every rank calls it at the same point with the same size.
struct PxRec {
    long long pid;
    unsigned long long host;
    unsigned long long ptr;
    int dev, ok;
    cudaIpcMemHandle_t h;
    char pad[128 - 32 - sizeof(cudaIpcMemHandle_t)];
};
static_assert(sizeof(PxRec) == 128, "PxRec is exchanged as 128 bytes");
static void px_unmap_peers(vbmf_b200_ctx* c) {
    auto& x = c->px;
    for (int r = 0; r < PX_MAX_WORLD; ++r) {
        if (x.ipc[r] && x.peer[r]) cudaIpcCloseMemHandle(x.peer[r]);
        x.peer[r] = nullptr; x.ipc[r] = false;
    }
}
static void px_release(vbmf_b200_ctx* c) {
    auto& x = c->px;
    px_unmap_peers(c);
    if (x.local) cudaFree(x.local);
    if (x.xchg) cudaFree(x.xchg);
    x.local = nullptr; x.xchg = nullptr; x.cap = 0; x.ok = false;
    cudaGetLastError();
}
static int px_setup(vbmf_b200_ctx* c, size_t data_bytes) {
    auto& x = c->px;
    if (c->world > PX_MAX_WORLD || x.failed || getenv("VBMF_B200_NO_PX") != nullptr) return 0;
    const size_t need = PX_FLAG_BYTES + data_bytes;
    if (x.ok && x.cap >= need) return 0;
    if (x.claimed) return 0;              // a live solver points into the buffer: it cannot be re-allocated now (the new solver uses NCCL)
    const int W = c->world;
    const size_t cap = (std::max(need, (size_t)32 << 20) + ((size_t)2 << 20) - 1) & ~(((size_t)2 << 20) - 1);
    if (W == 1) {
        // test switch VBMF_B200_PX_SELF=1: a single rank runs the exchange kernels against itself (same code, W = 1)
        if (getenv("VBMF_B200_PX_SELF") == nullptr) return 0;
        VB_CUDA_OK(cudaStreamSynchronize(c->st));
        px_release(c);
        if (cudaMalloc(&x.local, cap) != cudaSuccess) { cudaGetLastError(); x.local = nullptr; x.failed = true; return 0; }
        VB_CUDA_OK(cudaMemsetAsync(x.local, 0, cap, c->st));
        x.cap = cap; x.ok = true;
        return 0;
    }
    if (g_nccl.AllGather == nullptr) return 0;
    VB_CUDA_OK(cudaStreamSynchronize(c->st));
    if (x.local != nullptr && x.xchg != nullptr) {
        // growing: every rank unmaps its peers' buffers BEFORE any rank frees its own (an exported allocation must outlive
        // its imported mappings); a one-element all-reduce is the host-visible barrier between the two steps
        px_unmap_peers(c);
        double* dflag = (double*)(x.xchg + (size_t)(W + 1) * 128);
        VB_NCCL_OK(g_nccl.AllReduce(dflag, dflag, 1, /*ncclFloat64*/ 8, /*ncclSum*/ 0, c->comm, c->st));
        VB_CUDA_OK(cudaStreamSynchronize(c->st));
    }
    px_release(c);
    PxRec mine;
    memset(&mine, 0, sizeof(mine));
    mine.pid = (long long)getpid();
    {
        char hn[256] = "";
        gethostname(hn, sizeof(hn) - 1);
        unsigned long long hsh = 1469598103934665603ULL;
        for (const char* q = hn; *q; ++q) hsh = (hsh ^ (unsigned char)*q) * 1099511628211ULL;
        mine.host = hsh;
    }
    mine.dev = c->device;
    mine.ok = 1;
    if (cudaMalloc(&x.local, cap) != cudaSuccess || cudaMalloc(&x.xchg, (size_t)(W + 2) * 128) != cudaSuccess) { cudaGetLastError(); mine.ok = 0; }
    if (mine.ok && (cudaMemsetAsync(x.local, 0, cap, c->st) != cudaSuccess || cudaIpcGetMemHandle(&mine.h, x.local) != cudaSuccess)) { cudaGetLastError(); mine.ok = 0; }
    mine.ptr = (unsigned long long)(uintptr_t)x.local;
    if (x.xchg == nullptr) {      // nothing to exchange through: every rank must still take part in the collectives below
        if (cudaMalloc(&x.xchg, (size_t)(W + 2) * 128) != cudaSuccess) { cudaGetLastError(); set_error("cudaMalloc failed (peer exchange set-up)"); x.failed = true; return -1; }
    }
    std::vector<PxRec> all(W);
    VB_CUDA_OK(cudaMemcpyAsync(x.xchg, &mine, 128, cudaMemcpyHostToDevice, c->st));
    VB_NCCL_OK(g_nccl.AllGather(x.xchg, x.xchg + 128, 128, /*ncclInt8*/ 0, c->comm, c->st));
    VB_CUDA_OK(cudaMemcpyAsync(all.data(), x.xchg + 128, (size_t)W * 128, cudaMemcpyDeviceToHost, c->st));
    VB_CUDA_OK(cudaStreamSynchronize(c->st));
    int good = mine.ok;
    for (int r = 0; r < W && good; ++r) {
        if (r == c->rank) continue;
        const PxRec& pr = all[r];
        if (!pr.ok || pr.host != mine.host) { good = 0; break; }
        if (pr.pid == mine.pid) {
            int can = 0;
            if (pr.dev == c->device || cudaDeviceCanAccessPeer(&can, c->device, pr.dev) != cudaSuccess || !can) { cudaGetLastError(); good = 0; break; }
            const cudaError_t e = cudaDeviceEnablePeerAccess(pr.dev, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); good = 0; break; }
            cudaGetLastError();
            x.peer[r] = (char*)(uintptr_t)pr.ptr;
        } else {
            void* q = nullptr;
            if (cudaIpcOpenMemHandle(&q, pr.h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); good = 0; break; }
            x.peer[r] = (char*)q; x.ipc[r] = true;
        }
    }
    // agree: the number of ranks that could not map everybody
    double bad = good ? 0.0 : 1.0;
    double* dflag = (double*)(x.xchg + (size_t)(W + 1) * 128);
    VB_CUDA_OK(cudaMemcpyAsync(dflag, &bad, 8, cudaMemcpyHostToDevice, c->st));
    VB_NCCL_OK(g_nccl.AllReduce(dflag, dflag, 1, /*ncclFloat64*/ 8, /*ncclSum*/ 0, c->comm, c->st));
    VB_CUDA_OK(cudaMemcpyAsync(&bad, dflag, 8, cudaMemcpyDeviceToHost, c->st));
    VB_CUDA_OK(cudaStreamSynchronize(c->st));
    if (bad != 0.0) { px_release(c); x.failed = true; return 0; }
    x.cap = cap; x.ok = true;
    return 0;
}

extern "C" int vbmf_b200_version(void) { return 100; }
extern "C" const char* vbmf_b200_last_error(void) { return g_err; }
extern "C" int64_t vbmf_b200_launch_count(void) { return (int64_t)g_launches.load(); }
extern "C" int vbmf_b200_plan_contractions(int64_t L, int64_t M_local, int64_t H, int num_sms, int64_t* out6) {
    if (!out6 || L < 1 || M_local < 0 || H < 1 || H > 128 || num_sms < 1 || L > 0x7fffff00LL || M_local > 0x7fffff00LL) {
        set_error("plan_contractions: bad argument"); return -1;
    }
    int S1 = 1, kbs = 1, S2 = 1, kchunk = 16;
    plan_splitk_ytb((int)L, (int)M_local, (int)H, num_sms, &S1, &kbs);
    plan_splitk((int)L, (int)M_local, (int)H, num_sms, &S2, &kchunk);
    const GemmGeometry g = gemm_geometry((int)H);
    out6[0] = S1; out6[1] = kbs; out6[2] = S2; out6[3] = kchunk; out6[4] = g.ctas_per_sm; out6[5] = g.bn;
    return 0;
}
extern "C" int vbmf_b200_px_plan(int64_t L, int world, int rank, int64_t* out3) {
    if (!out3 || L < 1 || L > 0x7fffff00LL || world < 1 || world > PX_MAX_WORLD || rank < 0 || rank >= world) { set_error("px_plan: bad argument"); return -1; }
    int lo = 0, hi = 0, grid = 1;
    px_tile_range((int)L, world, rank, &lo, &hi, &grid);
    out3[0] = lo; out3[1] = hi; out3[2] = grid;
    return 0;
}
extern "C" int vbmf_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

extern "C" int vbmf_b200_nccl_unique_id(void* id128) {
    if (load_nccl()) return -1;
    NcclUniqueId id;
    VB_NCCL_OK(g_nccl.GetUniqueId(&id));
    memcpy(id128, &id, 128);
    return 0;
}

// comm_in: an already initialised communicator for this rank (single-process multi-device contexts, ncclCommInitAll) or NULL
static int ctx_create_impl(int device, int rank, int world, const void* nccl_id128, void* comm_in, void* cuda_stream,
                           vbmf_b200_ctx** out) {
    if (out == nullptr) { set_error("ctx_create: out is NULL"); return -1; }
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("no CUDA device available: vbmf_b200 has no CPU fallback");
        return -1;
    }
    if (device < 0 || device >= ndev) { set_error("device %d out of range (%d devices)", device, ndev); return -1; }
    VB_CUDA_OK(cudaSetDevice(device));
    cudaDeviceProp prop;
    VB_CUDA_OK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
        return -1;
    }
    if (gemm_init_device() || kernels_init_device()) return -1;      // per-device dynamic shared memory opt-ins
    vbmf_b200_ctx* c = new vbmf_b200_ctx();
    c->device = device; c->rank = rank; c->world = world < 1 ? 1 : world;
    c->num_sms = prop.multiProcessorCount;
    if (cuda_stream != nullptr) { c->st = (cudaStream_t)cuda_stream; c->own_stream = false; }
    else {
        if (cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking) != cudaSuccess) { set_error("cudaStreamCreate failed"); delete c; return -1; }
        c->own_stream = true;
    }
    const char* g = getenv("VBMF_B200_GEMM");
    c->simt = (g != nullptr && strcmp(g, "simt") == 0);
    c->gemm_dmma = (g != nullptr && strcmp(g, "dmma") == 0);
    if (c->world > 1) {
        if (comm_in != nullptr) c->comm = comm_in;
        else {
            if (nccl_id128 == nullptr) { set_error("world > 1 needs the NCCL unique id of rank 0"); delete c; return -1; }
            if (load_nccl()) { delete c; return -1; }
            NcclUniqueId id;
            memcpy(&id, nccl_id128, 128);
            int r = g_nccl.CommInitRank(&c->comm, c->world, id, rank);
            if (r != 0) { set_error("ncclCommInitRank failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?"); delete c; return -1; }
        }
    }
    if (cudaMalloc(&c->d_tr, 64) != cudaSuccess) { set_error("cudaMalloc failed"); delete c; return -1; }
    *out = c;
    return 0;
}
extern "C" int vbmf_b200_ctx_create(int device, int rank, int world, const void* nccl_id128, void* cuda_stream,
                                    vbmf_b200_ctx** out) {
    return ctx_create_impl(device, rank, world, nccl_id128, nullptr, cuda_stream, out);
}
// used by the single-process multi-device contexts (csrc/multi.cu)
namespace vb {
int ctx_create_with_comm(int device, int rank, int world, void* comm, vbmf_b200_ctx** out) {
    return ctx_create_impl(device, rank, world, nullptr, comm, nullptr, out);
}
int nccl_comm_init_all(void** comms, int ndev, const int* devs) {
    if (load_nccl()) return -1;
    if (!g_nccl.CommInitAll) { set_error("the NCCL library has no ncclCommInitAll"); return -1; }
    VB_NCCL_OK(g_nccl.CommInitAll(comms, ndev, devs));
    return 0;
}
}

static void ctx_free_Z(vbmf_b200_ctx* c) {
    if (c->Z) cudaFree(c->Z);
    if (c->Zexp) cudaFree(c->Zexp);
    c->Z = nullptr; c->Zexp = nullptr; c->Z_bytes = 0;
    c->z_ready = false; c->z_failed = false;
}

static void ctx_free_Y(vbmf_b200_ctx* c) {
    ctx_free_Z(c);
    if (c->copy_st) cudaStreamSynchronize(c->copy_st);
    if (c->stat_st) cudaStreamSynchronize(c->stat_st);
    c->chunks_pending = 0; c->tr_pending = false;
    if (c->Y) cudaFree(c->Y);
    if (c->rowY2) cudaFree(c->rowY2);
    if (c->stats_part) cudaFree(c->stats_part);
    c->Y = nullptr; c->rowY2 = nullptr; c->stats_part = nullptr; c->have_Y = false;
    c->Y_cap = 0; c->L_cap = 0;
}

extern "C" int vbmf_b200_ctx_destroy(vbmf_b200_ctx* c) {
    if (!c) return 0;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->st);
    ctx_free_Y(c);
    if (c->d_tr) cudaFree(c->d_tr);
    px_release(c);
    if (c->px.wait_ns) cudaFree(c->px.wait_ns);
    if (c->batch_dev) cudaFree(c->batch_dev);
    if (c->batch_host) cudaFreeHost(c->batch_host);
    for (auto e : c->ev_k1) cudaEventDestroy(e);
    for (auto e : c->ev_k2) cudaEventDestroy(e);
    for (auto e : c->ev_ar) cudaEventDestroy(e);
    for (auto& e : c->ev_seg) cudaEventDestroy(e.second);
    for (auto e : c->ev_chunk) cudaEventDestroy(e);
    if (c->ev_stats) cudaEventDestroy(c->ev_stats);
    if (c->copy_st) { cudaStreamSynchronize(c->copy_st); cudaStreamDestroy(c->copy_st); }
    if (c->stat_st) { cudaStreamSynchronize(c->stat_st); cudaStreamDestroy(c->stat_st); }
    if (c->comm) g_nccl.CommDestroy(c->comm);
    if (c->own_stream) cudaStreamDestroy(c->st);
    delete c;
    return 0;
}

extern "C" int vbmf_b200_ctx_sync(vbmf_b200_ctx* c) {
    VB_CUDA_OK(cudaSetDevice(c->device));
    if (c->copy_st) VB_CUDA_OK(cudaStreamSynchronize(c->copy_st));      // an asynchronous upload of Y, if any
    if (c->stat_st) VB_CUDA_OK(cudaStreamSynchronize(c->stat_st));
    VB_CUDA_OK(cudaStreamSynchronize(c->st));
    return 0;
}

static int ctx_alloc_Y(vbmf_b200_ctx* c, int64_t L, int64_t Mloc, int64_t Mglob, int64_t off) {
    if (L <= 0 || Mloc < 0 || Mglob < Mloc || off < 0 || off + Mloc > Mglob) { set_error("bad Y geometry L=%lld M_local=%lld M_global=%lld offset=%lld", (long long)L, (long long)Mloc, (long long)Mglob, (long long)off); return -1; }
    if (L > 0x7fffff00LL || Mglob > 0x7fffff00LL) { set_error("L and M must fit in 31 bits"); return -1; }
    VB_CUDA_OK(cudaSetDevice(c->device));
    VB_CUDA_OK(cudaStreamSynchronize(c->st));
    if (c->copy_st) VB_CUDA_OK(cudaStreamSynchronize(c->copy_st));
    if (c->stat_st) VB_CUDA_OK(cudaStreamSynchronize(c->stat_st));
    c->chunks_pending = 0; c->tr_pending = false;
    const int ld = (int)((L + 1) & ~1LL);                 // TMA needs a 16-byte pitch
    const size_t bytes = std::max<size_t>((size_t)ld * (size_t)std::max<int64_t>(Mloc, 1) * 8, 16);
    // Re-attaching a matrix of the same (or a somewhat smaller) size keeps the allocation: cudaFree + cudaMalloc of tens of
    // GB costs a few hundred ms, as much as the PCIe copy itself.  A much smaller matrix releases the big buffer.
    const bool reuse = c->Y != nullptr && c->rowY2 != nullptr && c->stats_part != nullptr && bytes <= c->Y_cap &&
                       c->Y_cap <= 2 * bytes + (64u << 20) && L <= c->L_cap;
    if (!reuse) {
        ctx_free_Y(c);
        VB_CUDA_OK(cudaMalloc(&c->Y, bytes));
        c->Y_cap = bytes;
        VB_CUDA_OK(cudaMalloc(&c->rowY2, (size_t)L * 8));
        VB_CUDA_OK(cudaMalloc(&c->stats_part, (size_t)(MAX_PARTS / 2) * L * 8));
        c->L_cap = (int)L;
    }
    c->have_Y = false;
    c->z_ready = false; c->z_failed = false;
    c->L = (int)L; c->Mloc = (int)Mloc; c->Mglob = (int)Mglob; c->moff = (int)off;
    c->ldY = ld;
    if (c->ldY != L) VB_CUDA_OK(cudaMemsetAsync(c->Y, 0, bytes, c->st));
    return 0;
}

static int ctx_finish_Y(vbmf_b200_ctx* c) {
    // tensor maps of the two contractions (K1 box 16 x 128, K2 box 16 x 16)
    if (c->Mloc > 0) {
        if (make_tmap_2d(&c->tmY1, c->Y, (uint64_t)c->L, (uint64_t)c->Mloc, (uint64_t)c->ldY * 8, 16, 128)) return -1;
        if (make_tmap_2d(&c->tmY2, c->Y, (uint64_t)c->L, (uint64_t)c->Mloc, (uint64_t)c->ldY * 8, 16, 16)) return -1;
    }
    // K0: row norms and trYTY
    Dev d;
    memset(&d, 0, sizeof(d));
    d.L = c->L; d.Mloc = c->Mloc; d.Y = c->Y; d.ldY = c->ldY; d.rowY2 = c->rowY2; d.part = c->stats_part;
    if (k_y_stats(c->st, d, c->d_tr)) return -1;
    if (c->world > 1) {
        if (ctx_allreduce(c, c->rowY2, (size_t)c->L)) return -1;
        if (k_total(c->st, c->rowY2, c->L, c->d_tr)) return -1;
    }
    VB_CUDA_OK(cudaMemcpyAsync(&c->trYTY, c->d_tr, 8, cudaMemcpyDeviceToHost, c->st));
    VB_CUDA_OK(cudaStreamSynchronize(c->st));
    c->have_Y = true;
    return 0;
}

// main stream ordered after the whole upload and K0; trYTY on the host when asked for
static int ctx_wait_upload(vbmf_b200_ctx* c) {
    if (c->chunks_pending > 0) {
        VB_CUDA_OK(cudaStreamWaitEvent(c->st, c->ev_stats, 0));
        c->chunks_pending = 0;
    }
    return 0;
}
static int ctx_host_trYTY(vbmf_b200_ctx* c) {
    if (c->tr_pending) {
        VB_CUDA_OK(cudaEventSynchronize(c->ev_stats));
        VB_CUDA_OK(cudaMemcpy(&c->trYTY, c->d_tr, 8, cudaMemcpyDeviceToHost));
        c->tr_pending = false;
    }
    return 0;
}
static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// The INT8 contractions run at H <= 64 unless the FP64 kernels are forced (VBMF_B200_GEMM=simt / dmma).
static bool ctx_int8_wanted(const vbmf_b200_ctx* c, int64_t H) {
    return !c->simt && !c->gemm_dmma && H >= 1 && H <= 64 && c->Y != nullptr && c->Mloc > 0;
}
// Slices of the resident Y, built on the main stream the first time an INT8 contraction needs them after Y changed (the
// caller has ordered the stream after the upload).  *ok = false when they cannot be allocated: the caller then runs the
// FP64 kernels.
static int ctx_slices(vbmf_b200_ctx* c, bool* ok) {
    *ok = false;
    if (c->z_failed || c->Y == nullptr || c->Mloc <= 0) return 0;
    if (c->z_ready) { *ok = true; return 0; }
    const int ldZ = i8_ld(c->L);
    const size_t bytes = (size_t)I8_NSL * c->Mloc * ldZ;
    // Zexp = F[L], E[Mloc], Fbad[L], Ebad[Mloc]; sized by ldZ >= L because a re-attach with the same Z_bytes may change L
    if (c->Z == nullptr || c->Z_bytes != bytes || c->ldZ != ldZ) {
        ctx_free_Z(c);
        if (cudaMalloc(&c->Z, bytes) != cudaSuccess || cudaMalloc(&c->Zexp, 2 * ((size_t)ldZ + c->Mloc) * 4) != cudaSuccess) {
            cudaGetLastError();
            ctx_free_Z(c);
            c->z_failed = true;
            return 0;
        }
        c->Z_bytes = bytes; c->ldZ = ldZ;
    }
    int* F = c->Zexp;
    if (i8_build_Y(c->st, c->Y, c->ldY, c->L, c->Mloc, c->Z, ldZ, F, F + c->L, F + c->L + c->Mloc, F + 2 * c->L + c->Mloc)) return -1;
    const uint64_t s1 = (uint64_t)ldZ, s2 = (uint64_t)ldZ * c->Mloc;
    if (make_tmap_3d_i8(&c->tmZ1, c->Z, (uint64_t)c->L, (uint64_t)c->Mloc, I8_NSL, s1, s2, 32, 128, I8_NSL, false)) return -1;
    if (make_tmap_3d_i8(&c->tmZ2, c->Z, (uint64_t)c->L, (uint64_t)c->Mloc, I8_NSL, s1, s2, 128, 32, I8_NSL, true)) return -1;
    c->z_ready = true;
    *ok = true;
    return 0;
}
// Split-K plans of the INT8 path: the FP64 plans with k ranges on multiples of 32 (K1: kbs1 16-row blocks per split)
static void i8_plans(int L, int M, int H, int num_sms, int* S1, int* kbs1, int* S, int* kchunk) {
    plan_splitk_ytb(L, M, H, num_sms, S1, kbs1);
    *kbs1 = (*kbs1 + 1) & ~1;
    const int nkb = (L + 15) / 16;
    *S1 = std::max(1, (nkb + *kbs1 - 1) / *kbs1);
    plan_splitk(L, M, H, num_sms, S, kchunk);
    *kchunk = (*kchunk + 31) / 32 * 32;
    *S = std::max(1, (M + *kchunk - 1) / *kchunk);
}
// operand digits of the INT8 path: K1 [I8_NSL][Hp][ldZ] + G[Hp], K2 [I8_NSL][Hp][ldM] + G[S][Hp] (one allocation)
struct I8Operands {
    char* mem = nullptr;
    uint8_t *Wb = nullptr, *Wa = nullptr;
    int *Gb = nullptr, *Ga = nullptr;
    int ldM = 0;
    CUtensorMap tmWb, tmWa;
    I8Operands() = default;
    I8Operands(const I8Operands&) = delete;
    I8Operands& operator=(const I8Operands&) = delete;
    ~I8Operands() { if (mem) cudaFree(mem); }
};
static int i8_operands_alloc(I8Operands* o, int L, int M, int H, int S, bool* ok) {
    *ok = false;
    const int Hp = i8_hpad(H), ldZ = i8_ld(L);
    o->ldM = i8_ld(std::max(M, 1));
    const size_t nb = align_up((size_t)I8_NSL * Hp * ldZ, 256), na = align_up((size_t)I8_NSL * Hp * o->ldM, 256);
    const size_t gb = align_up((size_t)Hp * 4, 256), ga = align_up((size_t)S * Hp * 4, 256);
    if (cudaMalloc(&o->mem, nb + na + gb + ga) != cudaSuccess) { cudaGetLastError(); o->mem = nullptr; return 0; }
    o->Wb = (uint8_t*)o->mem; o->Wa = o->Wb + nb; o->Gb = (int*)(o->Wa + na); o->Ga = (int*)((char*)o->Gb + gb);
    if (make_tmap_3d_i8(&o->tmWb, o->Wb, (uint64_t)L, (uint64_t)Hp, I8_NSL, (uint64_t)ldZ, (uint64_t)ldZ * Hp, 32, (uint32_t)Hp, I8_NSL, false)) return -1;
    if (M > 0 && make_tmap_3d_i8(&o->tmWa, o->Wa, (uint64_t)M, (uint64_t)Hp, I8_NSL, (uint64_t)o->ldM, (uint64_t)o->ldM * Hp, 32, (uint32_t)Hp, I8_NSL, false)) return -1;
    *ok = true;
    return 0;
}
// K1 on the INT8 path: P (or S1 slabs of it, stride M*H) = Y' * B
static int i8_k1(vbmf_b200_ctx* c, I8Operands* o, const double* B, int ldB, int H, double* P, int S1, int kbs1, const Scalars* sc) {
    const int* F = c->Zexp;
    const int* E = c->Zexp + c->L;
    const int* Ebad = c->Zexp + 2 * c->L + c->Mloc;
    if (i8_slice_B(c->st, B, ldB, c->L, H, F, o->Wb, c->ldZ, o->Gb, sc)) return -1;
    return launch_gemm_i8(c->st, false, &c->tmZ1, &o->tmWb, P, c->Mloc, c->L, S1, kbs1 * 16, H, E, Ebad, o->Gb, 0,
                          (size_t)c->Mloc * H, (size_t)H, 1, sc, c->num_sms);
}
// K2 on the INT8 path: S slabs [H][ldQ] of Y * A (A row-major [Mloc][H])
static int i8_k2(vbmf_b200_ctx* c, I8Operands* o, const double* A, int H, double* Qpart, int ldQ, int S, int kchunk, const Scalars* sc) {
    const int* F = c->Zexp;
    const int* E = c->Zexp + c->L;
    const int* Fbad = c->Zexp + c->L + c->Mloc;
    if (i8_slice_A(c->st, A, c->Mloc, H, E, kchunk, S, o->Wa, o->ldM, o->Ga, sc)) return -1;
    return launch_gemm_i8(c->st, true, &c->tmZ2, &o->tmWa, Qpart, c->L, c->Mloc, S, kchunk, H, F, Fbad, o->Ga, i8_hpad(H),
                          (size_t)H * ldQ, 1, (size_t)ldQ, sc, c->num_sms);
}

// Upload in column chunks on the copy stream, K0 chunk by chunk on the statistics stream; returns without waiting.
static int attach_Y_chunked(vbmf_b200_ctx* c, const double* Y, int64_t ldY, int64_t chunk_cols) {
    if (!c->copy_st) VB_CUDA_OK(cudaStreamCreateWithFlags(&c->copy_st, cudaStreamNonBlocking));
    if (!c->stat_st) VB_CUDA_OK(cudaStreamCreateWithFlags(&c->stat_st, cudaStreamNonBlocking));
    if (!c->ev_stats) VB_CUDA_OK(cudaEventCreateWithFlags(&c->ev_stats, cudaEventDisableTiming));
    c->chunk_c0.clear(); c->chunk_n.clear();
    for (int64_t c0 = 0; c0 < c->Mloc; c0 += chunk_cols) { c->chunk_c0.push_back((int)c0); c->chunk_n.push_back((int)std::min<int64_t>(chunk_cols, c->Mloc - c0)); }
    const size_t nch = c->chunk_c0.size();
    while (c->ev_chunk.size() < nch) { cudaEvent_t e; VB_CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); c->ev_chunk.push_back(e); }
    // the copy stream starts after whatever the main stream still does with the buffer (memset of the padding row)
    cudaEvent_t e0;
    VB_CUDA_OK(cudaEventCreateWithFlags(&e0, cudaEventDisableTiming));
    VB_CUDA_OK(cudaEventRecord(e0, c->st));
    VB_CUDA_OK(cudaStreamWaitEvent(c->copy_st, e0, 0));
    VB_CUDA_OK(cudaStreamWaitEvent(c->stat_st, e0, 0));
    VB_CUDA_OK(cudaEventDestroy(e0));
    Dev d;
    memset(&d, 0, sizeof(d));
    d.L = c->L; d.Mloc = c->Mloc; d.Y = c->Y; d.ldY = c->ldY; d.rowY2 = c->rowY2; d.part = c->stats_part;
    for (size_t k = 0; k < nch; ++k) {
        const size_t c0 = (size_t)c->chunk_c0[k], n = (size_t)c->chunk_n[k];
        if (ldY == c->L && c->ldY == c->L)
            VB_CUDA_OK(cudaMemcpyAsync(c->Y + c0 * c->ldY, Y + c0 * (size_t)ldY, (size_t)c->L * n * 8, cudaMemcpyHostToDevice, c->copy_st));
        else
            VB_CUDA_OK(cudaMemcpy2DAsync(c->Y + c0 * c->ldY, (size_t)c->ldY * 8, Y + c0 * (size_t)ldY, (size_t)ldY * 8, (size_t)c->L * 8, n,
                                         cudaMemcpyHostToDevice, c->copy_st));
        VB_CUDA_OK(cudaEventRecord(c->ev_chunk[k], c->copy_st));
        VB_CUDA_OK(cudaStreamWaitEvent(c->stat_st, c->ev_chunk[k], 0));
        if (k_y_stats_chunk(c->stat_st, d, (int)c0, (int)n, k == 0 ? 1 : 0)) return -1;
    }
    if (c->world > 1) VB_NCCL_OK(g_nccl.AllReduce(c->rowY2, c->rowY2, (size_t)c->L, 8, 0, c->comm, c->stat_st));
    if (k_total(c->stat_st, c->rowY2, c->L, c->d_tr)) return -1;
    VB_CUDA_OK(cudaEventRecord(c->ev_stats, c->stat_st));
    if (make_tmap_2d(&c->tmY1, c->Y, (uint64_t)c->L, (uint64_t)c->Mloc, (uint64_t)c->ldY * 8, 16, 128)) return -1;
    if (make_tmap_2d(&c->tmY2, c->Y, (uint64_t)c->L, (uint64_t)c->Mloc, (uint64_t)c->ldY * 8, 16, 16)) return -1;
    c->chunks_pending = (int)nch;
    c->tr_pending = true;
    c->trYTY = nan("");
    c->have_Y = true;
    return 0;
}

extern "C" int vbmf_b200_attach_Y(vbmf_b200_ctx* c, const double* Y, int64_t L, int64_t M_local, int64_t ldY,
                                  int64_t M_global, int64_t col_offset) {
    if (!c || (!Y && M_local > 0)) { set_error("attach_Y: NULL argument"); return -1; }
    if (ldY < L) { set_error("attach_Y: ldY < L"); return -1; }
    if (ctx_alloc_Y(c, L, M_local, M_global, col_offset)) return -1;
    {   // big matrices: chunked asynchronous upload (chunk = VBMF_B200_ATTACH_CHUNK_MB, default 2048 MB; at least two chunks)
        const char* e = getenv("VBMF_B200_ATTACH_CHUNK_MB");
        const double chunk_mb = e ? atof(e) : 2048.0;
        const double col_bytes = (double)c->ldY * 8.0;
        int64_t chunk_cols = (int64_t)(chunk_mb * 1048576.0 / col_bytes) / 128 * 128;
        if (chunk_cols < 128) chunk_cols = 128;
        if (chunk_mb > 0 && M_local >= 2 * chunk_cols && !c->simt) return attach_Y_chunked(c, Y, ldY, chunk_cols);
    }
    if (M_local > 0) {
        if (ldY == L && c->ldY == L) {       // contiguous on both sides: one plain copy (full PCIe rate from pinned memory)
            VB_CUDA_OK(cudaMemcpyAsync(c->Y, Y, (size_t)L * (size_t)M_local * 8, cudaMemcpyHostToDevice, c->st));
        } else {
            VB_CUDA_OK(cudaMemcpy2DAsync(c->Y, (size_t)c->ldY * 8, Y, (size_t)ldY * 8, (size_t)L * 8, (size_t)M_local,
                                         cudaMemcpyHostToDevice, c->st));
        }
    }
    return ctx_finish_Y(c);
}

extern "C" int vbmf_b200_set_shape(vbmf_b200_ctx* c, int64_t L, int64_t M_local, int64_t M_global, int64_t col_offset) {
    if (!c) { set_error("set_shape: NULL ctx"); return -1; }
    if (L <= 0 || M_local < 0 || M_global < M_local || col_offset < 0 || col_offset + M_local > M_global || L > 0x7fffff00LL || M_global > 0x7fffff00LL) {
        set_error("set_shape: bad geometry"); return -1;
    }
    VB_CUDA_OK(cudaSetDevice(c->device));
    VB_CUDA_OK(cudaStreamSynchronize(c->st));
    ctx_free_Y(c);
    c->L = (int)L; c->Mloc = (int)M_local; c->Mglob = (int)M_global; c->moff = (int)col_offset;
    c->ldY = (int)((L + 1) & ~1LL);
    c->trYTY = nan("");
    c->have_Y = true;          // geometry only: Y stays NULL, steps that contract with Y refuse to run
    return 0;
}

extern "C" int vbmf_b200_synth_Y(vbmf_b200_ctx* c, int64_t L, int64_t M_local, int64_t M_global, int64_t col_offset,
                                 int rank, double noise, uint64_t seed) {
    if (!c) { set_error("synth_Y: NULL ctx"); return -1; }
    if (ctx_alloc_Y(c, L, M_local, M_global, col_offset)) return -1;
    if (k_synth(c->st, c->Y, c->ldY, c->L, c->Mloc, c->moff, rank, noise, seed)) return -1;
    return ctx_finish_Y(c);
}

extern "C" int vbmf_b200_preprocess_Y(vbmf_b200_ctx* c, double lambda, int64_t* L_out, int64_t* used_rows) {
    if (!c || !c->have_Y || !c->Y) { set_error("preprocess_Y: no Y attached"); return -1; }
    VB_CUDA_OK(cudaSetDevice(c->device));
    if (ctx_wait_upload(c) || ctx_host_trYTY(c)) return -1;
    const int L = c->L, M = c->Mloc;
    cudaStream_t st = c->st;
    double *mu = nullptr, *den = nullptr, *rs = nullptr;
    VB_CUDA_OK(cudaMalloc(&mu, (size_t)L * 8));
    VB_CUDA_OK(cudaMalloc(&den, (size_t)L * 8));
    VB_CUDA_OK(cudaMalloc(&rs, (size_t)L * 8));
    int rc = 0;
    // mean(Y, 2) and var(Y, 2) over ALL columns (all-reduced across shards), src/util.jl:38-39
    rc = k_row_pass(st, c->Y, c->ldY, L, M, 0, nullptr, nullptr, c->stats_part, mu);
    if (!rc) rc = ctx_allreduce(c, mu, (size_t)L);
    if (!rc) rc = k_finish_stats(st, mu, L, (double)c->Mglob, 0);
    if (!rc) rc = k_row_pass(st, c->Y, c->ldY, L, M, 1, mu, nullptr, c->stats_part, den);
    if (!rc) rc = ctx_allreduce(c, den, (size_t)L);
    if (!rc) rc = k_finish_stats(st, den, L, (double)c->Mglob, 1);
    // scale in place, rowsums = sum(abs(sY), 2), src/util.jl:75-76
    if (!rc) rc = k_row_pass(st, c->Y, c->ldY, L, M, 2, mu, den, c->stats_part, rs);
    if (!rc) rc = ctx_allreduce(c, rs, (size_t)L);
    std::vector<double> hrs((size_t)L);
    if (!rc && cudaMemcpyAsync(hrs.data(), rs, (size_t)L * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess) { set_error("preprocess_Y: copy failed"); rc = -1; }
    if (!rc && cudaStreamSynchronize(st) != cudaSuccess) { set_error("preprocess_Y: sync failed"); rc = -1; }
    cudaFree(mu); cudaFree(den); cudaFree(rs);
    if (rc) return rc;
    std::vector<int> rows;
    for (int l = 0; l < L; ++l) if (hrs[l] >= 1e-5) rows.push_back(l);      // used_rows[rowsums .>= 1e-5], :79
    const int Lnew = (int)rows.size();
    if (Lnew == 0) { set_error("preprocess_Y: every row is constant, nothing left"); return -1; }
    c->z_ready = false; c->z_failed = false;
    if (Lnew == L) {
        if (k_scale_all(st, c->Y, (size_t)c->ldY * (size_t)std::max(M, 1), lambda)) return -1;
    } else {
        const int ldn = (Lnew + 1) & ~1;
        double* Yn = nullptr;
        int* drows = nullptr;
        const size_t bytes = std::max<size_t>((size_t)ldn * (size_t)std::max(M, 1) * 8, 16);
        VB_CUDA_OK(cudaMalloc(&Yn, bytes));
        VB_CUDA_OK(cudaMalloc(&drows, (size_t)Lnew * 4));
        VB_CUDA_OK(cudaMemsetAsync(Yn, 0, bytes, st));
        VB_CUDA_OK(cudaMemcpyAsync(drows, rows.data(), (size_t)Lnew * 4, cudaMemcpyHostToDevice, st));
        if (k_compact_rows(st, c->Y, c->ldY, Yn, ldn, drows, Lnew, M, lambda)) return -1;
        VB_CUDA_OK(cudaStreamSynchronize(st));
        cudaFree(drows);
        cudaFree(c->Y);                       // rowY2 / stats_part were sized for the larger L and are kept
        c->Y = Yn; c->Y_cap = bytes; c->L = Lnew; c->ldY = ldn;
    }
    if (L_out) *L_out = Lnew;
    if (used_rows) for (int k = 0; k < Lnew; ++k) used_rows[k] = rows[k] + 1;
    return ctx_finish_Y(c);
}

extern "C" int vbmf_b200_download_Y(vbmf_b200_ctx* c, double* out, int64_t ldY) {
    if (!c || !c->have_Y || !c->Y) { set_error("download_Y: no Y attached"); return -1; }
    VB_CUDA_OK(cudaSetDevice(c->device));
    if (ctx_wait_upload(c)) return -1;
    if (c->Mloc > 0)
        VB_CUDA_OK(cudaMemcpy2DAsync(out, (size_t)ldY * 8, c->Y, (size_t)c->ldY * 8, (size_t)c->L * 8, (size_t)c->Mloc,
                                     cudaMemcpyDeviceToHost, c->st));
    VB_CUDA_OK(cudaStreamSynchronize(c->st));
    return 0;
}

extern "C" int vbmf_b200_trYTY(vbmf_b200_ctx* c, double* out) {
    if (!c || !c->have_Y) { set_error("trYTY: no Y attached"); return -1; }
    if (ctx_host_trYTY(c)) return -1;
    *out = c->trYTY;
    return 0;
}

extern "C" int vbmf_b200_ctx_profile(vbmf_b200_ctx* c, int enable) {
    c->profile = (enable & 1) != 0;
    c->profile_segments = c->profile && (enable & 2) != 0;
    if (c->profile_segments && c->px.wait_ns == nullptr) {
        VB_CUDA_OK(cudaSetDevice(c->device));
        if (cudaMalloc(&c->px.wait_ns, 256) != cudaSuccess) { cudaGetLastError(); c->px.wait_ns = nullptr; }
    }
    if (c->px.wait_ns) cudaMemsetAsync(c->px.wait_ns, 0, 256, c->st);
    for (auto e : c->ev_k1) cudaEventDestroy(e);
    for (auto e : c->ev_k2) cudaEventDestroy(e);
    for (auto e : c->ev_ar) cudaEventDestroy(e);
    for (auto& e : c->ev_seg) cudaEventDestroy(e.second);
    c->ev_k1.clear(); c->ev_k2.clear(); c->ev_ar.clear(); c->ev_seg.clear();
    return 0;
}
// CUDA-event time of the per-iteration all-reduce launches (world > 1; zero launches otherwise)
extern "C" int vbmf_b200_ctx_peer_exchange(vbmf_b200_ctx* c) { return (c != nullptr && c->px.ok) ? 1 : 0; }
extern "C" int vbmf_b200_ctx_profile_read_allreduce(vbmf_b200_ctx* c, double* ar_ms, int64_t* ar_n) {
    VB_CUDA_OK(cudaStreamSynchronize(c->st));
    double t = 0;
    for (size_t i = 0; i + 1 < c->ev_ar.size(); i += 2) { float ms = 0; VB_CUDA_OK(cudaEventElapsedTime(&ms, c->ev_ar[i], c->ev_ar[i + 1])); t += ms; }
    *ar_ms = t; *ar_n = (int64_t)(c->ev_ar.size() / 2);
    return 0;
}
extern "C" int vbmf_b200_ctx_profile_read(vbmf_b200_ctx* c, double* k1_ms, int64_t* k1_n, double* k2_ms, int64_t* k2_n) {
    VB_CUDA_OK(cudaStreamSynchronize(c->st));
    double t1 = 0, t2 = 0;
    for (size_t i = 0; i + 1 < c->ev_k1.size(); i += 2) { float ms = 0; VB_CUDA_OK(cudaEventElapsedTime(&ms, c->ev_k1[i], c->ev_k1[i + 1])); t1 += ms; }
    for (size_t i = 0; i + 1 < c->ev_k2.size(); i += 2) { float ms = 0; VB_CUDA_OK(cudaEventElapsedTime(&ms, c->ev_k2[i], c->ev_k2[i + 1])); t2 += ms; }
    *k1_ms = t1; *k1_n = (int64_t)(c->ev_k1.size() / 2); *k2_ms = t2; *k2_n = (int64_t)(c->ev_k2.size() / 2);
    return 0;
}
// Segment marks of one iteration on the main stream (profiling only): the time since the previous mark is booked on `tag`.
enum { SEG_START = 0, SEG_K1, SEG_A_EPI, SEG_K2, SEG_REDUCE_Q, SEG_EXCHANGE, SEG_SIGMA_B, SEG_B_EPI, SEG_B_REDUCE,
       SEG_WAIT_SMALL, SEG_WAIT_EPI, SEG_WAIT_REDUCE,                // mean barrier wait of CTA 0 (peer exchange)
       SEG_PH0, SEG_COUNT = SEG_PH0 + 9 };                           // phases of CTA 0 in the last epilogue / Gram reduction launch
static void prof_seg(vbmf_b200_ctx* c, int tag) {
    if (!c->profile_segments) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) == cudaSuccess) { cudaEventRecord(e, c->st); c->ev_seg.emplace_back(tag, e); }
}
extern "C" int vbmf_b200_ctx_profile_read_segments(vbmf_b200_ctx* c, double* ms, int64_t* n, int cap) {
    if (!c || !ms || !n) { set_error("NULL argument"); return -1; }
    VB_CUDA_OK(cudaStreamSynchronize(c->st));
    for (int i = 0; i < cap; ++i) { ms[i] = 0.0; n[i] = 0; }
    for (size_t i = 1; i < c->ev_seg.size(); ++i) {
        const int tag = c->ev_seg[i].first;
        if (tag == SEG_START || tag >= cap) continue;
        float t = 0;
        VB_CUDA_OK(cudaEventElapsedTime(&t, c->ev_seg[i - 1].second, c->ev_seg[i].second));
        ms[tag] += t; n[tag] += 1;
    }
    if (c->px.wait_ns != nullptr && cap >= SEG_COUNT) {
        unsigned long long w[6] = {0, 0, 0, 0, 0, 0};
        VB_CUDA_OK(cudaMemcpy(w, c->px.wait_ns, sizeof(w), cudaMemcpyDeviceToHost));
        for (int k = 0; k < 3; ++k) { ms[SEG_WAIT_SMALL + k] = (double)w[2 * k] * 1e-6; n[SEG_WAIT_SMALL + k] = (int64_t)w[2 * k + 1]; }
        unsigned long long ph[12];
        VB_CUDA_OK(cudaMemcpy(ph, c->px.wait_ns + 8, sizeof(ph), cudaMemcpyDeviceToHost));
        // epilogue: SigmaB fill, barrier, Q loads, product + stores, Gram, partial out; reduction: local sum, push + barrier, final
        const int from[9] = {0, 1, 2, 3, 4, 5, 8, 9, 10}, to[9] = {1, 2, 3, 4, 5, 6, 9, 10, 11};
        for (int k = 0; k < 9; ++k) if (ph[to[k]] >= ph[from[k]] && ph[from[k]] != 0) { ms[SEG_PH0 + k] = (double)(ph[to[k]] - ph[from[k]]) * 1e-6; n[SEG_PH0 + k] = 1; }
    }
    return SEG_COUNT;
}
static void prof_mark(vbmf_b200_ctx* c, std::vector<cudaEvent_t>& v) {
    if (!c->profile) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) == cudaSuccess) { cudaEventRecord(e, c->st); v.push_back(e); }
}

// ------------------------------------------------------------------------------------------- solver
struct vbmf_b200_solver {
    vbmf_b200_ctx* c = nullptr;
    Dev d;
    char* arena = nullptr;
    size_t arena_bytes = 0;
    double* Qpart = nullptr;
    int S = 1, kchunk = 16;
    double* Ppart = nullptr;      // split-K slabs of K1 (nullptr when S1 == 1)
    int S1 = 1, kbs1 = 1;
    int* d_labels = nullptr;
    CUtensorMap tmB, tmBs, tmA;
    bool k2_simt = false;
    bool i8 = false;              // K1 / K2 on the INT8 tensor cores (gemm_int8.cu) whenever Y's slices are available
    I8Operands i8o;
    // host-side validity of derived quantities (every enqueued kernel either runs or is skipped as a whole iteration)
    bool btb_valid = false, ata_valid = false, q_valid = false, extras_valid = false, mean_valid = false;
    bool ata_local = false;   // packed.AtA holds this shard's AHat'AHat (not yet all-reduced)
    int ata_parts = 0;        // > 0: ... as soon as that many Gram partials in d.part are summed (deferred to the side stream, beside K2)
    int diag_parts = 0;       // > 0: the fused diagonal pass left that many partials (A'A | column sums | group sums) in d.part, same deferral
    bool ca_done = false;     // the fused diagonal A pass already did updateCA! of this iteration
    bool loop_ahead = false;      // set by solver_run while it enqueues whole iterations back to back
    bool sigmaA_ahead = false;    // dense loop: the NEXT iteration's SigmaA was already inverted on the side stream (behind post)
    bool need_tr_copy = false;    // dense: sum(Y.^2) was still being computed at upload time; copy it device-side before its first use
    double* Qc = nullptr;         // [chunks][H*ldB] per-chunk Y*AHat of the upload-overlapped first iteration (allocated on demand)
    size_t Qc_chunks = 0;
    int S_chunk = 1;              // K2 slabs of the largest upload chunk (Qpart is sized for max(S, S_chunk))
    int* h_flag = nullptr;   // pinned, 2 slots
    cudaEvent_t ev[2] = {nullptr, nullptr};
    // The single-CTA tail of an iteration (norms, hyper-parameter updates, convergence test) runs on a side stream so that
    // the next iteration's K1 -- which only needs BHat -- starts right behind the B epilogue instead of waiting for it.
    cudaStream_t side = nullptr;
    cudaEvent_t ev_b = nullptr, ev_p = nullptr;
    bool post_pending = false;
    // small problems are launch bound: one iteration is captured into a CUDA graph and replayed
    cudaGraphExec_t gexec = nullptr;
    int gexec_flags = -1;
    // peer exchange: packed / BHat / rank partials live in the context's peer-visible buffer at these byte offsets
    bool px = false;
    size_t px_packed = 0, px_B = 0, px_gpart = 0, px_small = 0;
    cudaEvent_t ev_a = nullptr, ev_sb = nullptr;   // A side of the iteration done (main) -> small exchange + SigmaB (side) -> epilogue (main)
    Scalars h_sc;
};


static int solver_create_impl(vbmf_b200_ctx* c, int kind, int64_t H, int64_t h_split, int64_t M0_global, int64_t n_labels,
                              const int64_t* labels, int keep_blocks, vbmf_b200_solver** out) {
    if (out == nullptr) { set_error("solver_create: out is NULL"); return -1; }
    *out = nullptr;
    if (!c || !c->have_Y) { set_error("solver_create: attach Y first"); return -1; }
    if (kind < 0 || kind > 3) { set_error("solver_create: unknown kind %d", kind); return -1; }
    if (kind == VBMF_B200_TRIAL && (M0_global < 0 || M0_global > c->Mglob)) { set_error("M0 must be in 0..M"); return -1; }
    if (H < 1 || H > 128) { set_error("H = %lld is outside the supported range 1..128", (long long)H); return -1; }
    const bool grouped = kind == VBMF_B200_DUAL || kind == VBMF_B200_TRIAL;
    if (grouped && (h_split < 0 || h_split > H)) { set_error("H must be at least H0!"); return -1; }  // src/vbmf_dual.jl:126-128
    if (!grouped && (h_split < 0 || h_split > H)) { set_error("H1 must be in 0..H"); return -1; }
    VB_CUDA_OK(cudaSetDevice(c->device));
    vbmf_b200_solver* s = new vbmf_b200_solver();
    s->c = c;
    Dev& d = s->d;
    memset(&d, 0, sizeof(d));
    d.kind = kind;
    d.L = c->L; d.ldB = (c->L + 1) & ~1;
    d.Mloc = c->Mloc; d.Mglob = c->Mglob; d.moff = c->moff;
    d.H = (int)H;
    if (grouped) { d.H0 = (int)h_split; d.H1 = (int)(H - h_split); }
    else { d.H0 = (int)H; d.H1 = (int)h_split; }
    d.M0 = (kind == VBMF_B200_TRIAL) ? (int)M0_global : c->Mglob;
    d.nlabels = grouped ? 0 : (int)n_labels;
    d.Y = c->Y; d.ldY = c->ldY; d.rowY2 = c->rowY2;

    plan_splitk(d.L, d.Mloc, d.H, c->num_sms, &s->S, &s->kchunk);
    plan_splitk_ytb(d.L, d.Mloc, d.H, c->num_sms, &s->S1, &s->kbs1);
    if (c->simt) s->S1 = 1;
    s->i8 = ctx_int8_wanted(c, H);
    if (s->i8) {
        i8_plans(d.L, d.Mloc, d.H, c->num_sms, &s->S1, &s->kbs1, &s->S, &s->kchunk);
        if (i8_operands_alloc(&s->i8o, d.L, d.Mloc, d.H, s->S, &s->i8)) { delete s; return -1; }
    }
    if (c->chunks_pending > 0 && kind == VBMF_B200_DENSE) {      // the first iteration may run chunk by chunk behind the upload
        for (size_t k = 0; k < c->chunk_n.size(); ++k) {
            int Sc = 1, kc = 16;
            plan_splitk(d.L, c->chunk_n[k], d.H, c->num_sms, &Sc, &kc);
            s->S_chunk = std::max(s->S_chunk, Sc);
        }
    }
    s->k2_simt = c->simt || (H % 2 != 0);       // the A tensor map needs a 16-byte row pitch

    const size_t MH = (size_t)std::max(d.Mloc, 1) * H, LH = (size_t)H * d.ldB, HH = (size_t)H * H, Lr = (size_t)d.L;
    const size_t part_elems = std::max<size_t>({(size_t)MAX_PARTS * HH, (size_t)2400 * std::min<size_t>(H, 32) * std::min<size_t>(H, 32),
                                                (size_t)300 * Lr, (size_t)16384});
    // world > 1, H <= 64: the updateB! exchange runs through peer-mapped memory (kernels.cuh, PxDev); the payload and BHat then
    // live in the context's peer-visible buffer.  One solver per context at a time owns it; the others use the NCCL all-reduce.
    if ((c->world > 1 || getenv("VBMF_B200_PX_SELF") != nullptr) && H <= 64) {
        s->px_packed = PX_FLAG_BYTES;
        s->px_B = s->px_packed + align_up((LH + 2 * HH + 8) * 8, 256);
        s->px_gpart = s->px_B + align_up(LH * 8, 256);
        s->px_small = s->px_gpart + align_up((size_t)PX_MAX_WORLD * (2 * HH + 1) * 8, 256);
        const size_t px_end = s->px_small + align_up((2 * HH + 8) * 8, 256);
        if (px_setup(c, px_end - PX_FLAG_BYTES)) { delete s; return -1; }
        if (c->px.ok && !c->px.claimed) {
            s->px = true; c->px.claimed = true;
            if (cudaMemsetAsync(c->px.local + PX_FLAG_BYTES, 0, px_end - PX_FLAG_BYTES, c->st) != cudaSuccess) { set_error("cudaMemset failed"); c->px.claimed = false; delete s; return -1; }
        }
    }
    struct Item { double** p; size_t n; };
    std::vector<Item> items = {
        {&d.A, MH}, {&d.P, MH}, {&d.Bold, LH}, {&d.D, LH}, {&d.Bs, LH},
        {&d.SigmaA, HH}, {&d.SigmaB, HH}, {&d.BtB, HH}, {&d.BtBw, HH}, {&d.DtD, HH}, {&d.Gm, HH},
        {&d.sigmaVec, Lr}, {&d.etaVec, Lr}, {&d.zetaVec, Lr}, {&d.part, part_elems}, {&d.lbacc, 32},
        {&s->Qpart, (size_t)std::max(s->S, s->S_chunk) * LH},
    };
    if (s->S1 > 1) items.push_back({&s->Ppart, (size_t)s->S1 * MH});
    if (s->px) {
        d.packed = (double*)(c->px.local + s->px_packed);
        d.B = (double*)(c->px.local + s->px_B);
    } else { items.push_back({&d.B, LH}); items.push_back({&d.packed, LH + 2 * HH + 8}); }
    if (kind == VBMF_B200_DENSE) { items.push_back({&d.CA, HH}); items.push_back({&d.CB, HH}); items.push_back({&d.invCA, HH}); items.push_back({&d.invCB, HH}); }
    else {
        items.push_back({&d.CAv, MH}); items.push_back({&d.beta, MH}); items.push_back({&d.sdiag, MH});
        items.push_back({&d.CBv, (size_t)H}); items.push_back({&d.deltav, (size_t)H});
        if (keep_blocks) items.push_back({&d.blocks, MH * H});
    }
    size_t total = 256 + align_up(sizeof(Scalars), 256) + align_up((size_t)std::max(d.nlabels, 1) * 4, 256) + align_up((size_t)std::max(d.Mloc, 1), 256);
    for (auto& it : items) total += align_up(it.n * 8, 256);
    if (cudaMalloc(&s->arena, total) != cudaSuccess) {
        cudaGetLastError();
        set_error("cudaMalloc of %zu bytes of solver state failed", total);
        if (s->px) c->px.claimed = false;
        delete s;
        return -1;
    }
    s->arena_bytes = total;
    if (cudaMemsetAsync(s->arena, 0, total, c->st) != cudaSuccess) { set_error("cudaMemset failed"); cudaFree(s->arena); if (s->px) c->px.claimed = false; delete s; return -1; }
    char* p = s->arena;
    d.sc = (Scalars*)p; p += align_up(sizeof(Scalars), 256);
    s->d_labels = (int*)p; p += align_up((size_t)std::max(d.nlabels, 1) * 4, 256);
    unsigned char* d_rowmask = (unsigned char*)p; p += align_up((size_t)std::max(d.Mloc, 1), 256);
    for (auto& it : items) { *it.p = (double*)p; p += align_up(it.n * 8, 256); }
    d.labels = s->d_labels;
    if (d.nlabels > 0) {
        std::vector<int> lab(d.nlabels);
        for (int i = 0; i < d.nlabels; ++i) {
            const int64_t v = labels[i];
            if (v < 1 || v > d.Mloc) { set_error("label %lld out of range 1..%d", (long long)v, d.Mloc); cudaFree(s->arena); if (s->px) c->px.claimed = false; delete s; return -1; }
            lab[i] = (int)(v - 1);
        }
        std::vector<unsigned char> rm((size_t)std::max(d.Mloc, 1), 0);
        for (int v : lab) rm[v] = 1;
        if (cudaMemcpyAsync(s->d_labels, lab.data(), (size_t)d.nlabels * 4, cudaMemcpyHostToDevice, c->st) != cudaSuccess ||
            cudaMemcpyAsync(d_rowmask, rm.data(), rm.size(), cudaMemcpyHostToDevice, c->st) != cudaSuccess ||
            cudaStreamSynchronize(c->st) != cudaSuccess) { set_error("label upload failed"); cudaFree(s->arena); if (s->px) c->px.claimed = false; delete s; return -1; }
        d.rowmask = (d.H1 > 0) ? d_rowmask : nullptr;
    }
    const GemmGeometry g = gemm_geometry(d.H);
    int rc = 0;
    rc |= make_tmap_2d(&s->tmB, d.B, (uint64_t)d.L, (uint64_t)H, (uint64_t)d.ldB * 8, 16, (uint32_t)g.bn);
    rc |= make_tmap_2d(&s->tmBs, d.Bs, (uint64_t)d.L, (uint64_t)H, (uint64_t)d.ldB * 8, 16, (uint32_t)g.bn);
    if (!s->k2_simt && d.Mloc > 0) rc |= make_tmap_2d(&s->tmA, d.A, (uint64_t)H, (uint64_t)d.Mloc, (uint64_t)H * 8, 16, 16);
    if (rc) { cudaFree(s->arena); if (s->px) c->px.claimed = false; delete s; return -1; }
    if (cudaMallocHost(&s->h_flag, 2 * sizeof(int)) != cudaSuccess || cudaEventCreateWithFlags(&s->ev[0], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev[1], cudaEventDisableTiming) != cudaSuccess ||
        cudaStreamCreateWithFlags(&s->side, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_b, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_p, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_a, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_sb, cudaEventDisableTiming) != cudaSuccess) {
        set_error("pinned flag / event allocation failed"); cudaFree(s->arena); if (s->px) c->px.claimed = false; delete s; return -1;
    }
    memset(&s->h_sc, 0, sizeof(Scalars));
    *out = s;
    return 0;
}

extern "C" int vbmf_b200_solver_create(vbmf_b200_ctx* c, int kind, int64_t H, int64_t h_split, int64_t n_labels,
                                       const int64_t* labels, int keep_blocks, vbmf_b200_solver** out) {
    if (kind == VBMF_B200_TRIAL) { set_error("use vbmf_b200_solver_create_trial for vbmf_trial parameters"); return -1; }
    return solver_create_impl(c, kind, H, h_split, 0, n_labels, labels, keep_blocks, out);
}
extern "C" int vbmf_b200_solver_create_trial(vbmf_b200_ctx* c, int64_t H, int64_t H0, int64_t M0_global, int keep_blocks,
                                             vbmf_b200_solver** out) {
    return solver_create_impl(c, VBMF_B200_TRIAL, H, H0, M0_global, 0, nullptr, keep_blocks, out);
}

extern "C" int vbmf_b200_solver_destroy(vbmf_b200_solver* s) {
    if (!s) return 0;
    cudaSetDevice(s->c->device);
    cudaStreamSynchronize(s->c->st);
    if (s->side) { cudaStreamSynchronize(s->side); cudaStreamDestroy(s->side); }
    if (s->gexec) cudaGraphExecDestroy(s->gexec);
    if (s->ev_b) cudaEventDestroy(s->ev_b);
    if (s->ev_p) cudaEventDestroy(s->ev_p);
    if (s->ev_a) cudaEventDestroy(s->ev_a);
    if (s->ev_sb) cudaEventDestroy(s->ev_sb);
    if (s->arena) cudaFree(s->arena);
    if (s->Qc) cudaFree(s->Qc);
    if (s->h_flag) cudaFreeHost(s->h_flag);
    for (int i = 0; i < 2; ++i) if (s->ev[i]) cudaEventDestroy(s->ev[i]);
    if (s->px) s->c->px.claimed = false;
    delete s;
    return 0;
}

// ---- host <-> device marshalling -------------------------------------------------------------------------------------
static int up(vbmf_b200_solver* s, double* dst, const double* src, size_t n) {
    if (n == 0) return 0;
    if (src == nullptr) { set_error("upload: a required array pointer is NULL"); return -1; }
    VB_CUDA_OK(cudaMemcpyAsync(dst, src, n * 8, cudaMemcpyHostToDevice, s->c->st));
    return 0;
}
static int down(vbmf_b200_solver* s, double* dst, const double* src, size_t n) {
    if (n == 0 || dst == nullptr) return 0;
    VB_CUDA_OK(cudaMemcpyAsync(dst, src, n * 8, cudaMemcpyDeviceToHost, s->c->st));
    return 0;
}
static int up_B(vbmf_b200_solver* s, const double* BHat) {
    if (BHat == nullptr) { set_error("upload: BHat is NULL"); return -1; }
    const Dev& d = s->d;
    VB_CUDA_OK(cudaMemcpy2DAsync(d.B, (size_t)d.ldB * 8, BHat, (size_t)d.L * 8, (size_t)d.L * 8, (size_t)d.H, cudaMemcpyHostToDevice, s->c->st));
    return 0;
}
static int down_B(vbmf_b200_solver* s, double* BHat) {
    if (BHat == nullptr) return 0;
    const Dev& d = s->d;
    VB_CUDA_OK(cudaMemcpy2DAsync(BHat, (size_t)d.L * 8, d.B, (size_t)d.ldB * 8, (size_t)d.L * 8, (size_t)d.H, cudaMemcpyDeviceToHost, s->c->st));
    return 0;
}
// AHat (M x H column-major, Julia) -> A ([M][H] rows); P is the staging buffer
static int up_A(vbmf_b200_solver* s, const double* AHat, const double* ATVecHat) {
    const Dev& d = s->d;
    const size_t n = (size_t)d.Mloc * d.H;
    if (ATVecHat != nullptr) return up(s, d.A, ATVecHat, n);
    if (up(s, d.P, AHat, n)) return -1;
    return k_transpose(s->c->st, d.P, d.A, d.Mloc, d.H);
}
static int down_A(vbmf_b200_solver* s, double* AHat, double* ATVecHat) {
    const Dev& d = s->d;
    const size_t n = (size_t)d.Mloc * d.H;
    if (down(s, ATVecHat, d.A, n)) return -1;
    if (AHat != nullptr) {
        if (k_transpose(s->c->st, d.A, d.P, d.H, d.Mloc)) return -1;     // A viewed as column-major H x M
        if (down(s, AHat, d.P, n)) return -1;
    }
    return 0;
}
static int push_scalars(vbmf_b200_solver* s) {
    s->h_sc.active = 0;
    s->h_sc.chol_fail = 0;
    VB_CUDA_OK(cudaMemcpyAsync(s->d.sc, &s->h_sc, sizeof(Scalars), cudaMemcpyHostToDevice, s->c->st));
    VB_CUDA_OK(cudaStreamSynchronize(s->c->st));
    s->btb_valid = s->ata_valid = s->q_valid = s->extras_valid = s->mean_valid = s->ata_local = false;
    return 0;
}
static int pull_scalars(vbmf_b200_solver* s) {
    VB_CUDA_OK(cudaMemcpyAsync(&s->h_sc, s->d.sc, sizeof(Scalars), cudaMemcpyDeviceToHost, s->c->st));
    VB_CUDA_OK(cudaStreamSynchronize(s->c->st));
    return 0;
}
static int check_dims(vbmf_b200_solver* s, int kind, int64_t L, int64_t M, int64_t H) {
    const Dev& d = s->d;
    if (d.kind != kind) { set_error("state struct kind does not match the solver"); return -1; }
    if (L != d.L || M != d.Mloc || H != d.H) {
        set_error("state dims (L=%lld, M=%lld, H=%lld) do not match the solver (L=%d, M=%d, H=%d)", (long long)L, (long long)M, (long long)H, d.L, d.Mloc, d.H);
        return -1;
    }
    return 0;
}
static int down_yhat(vbmf_b200_solver* s, double* YHat) {
    if (YHat == nullptr) return 0;
    return vbmf_b200_solver_yhat(s, YHat, s->d.L);
}

extern "C" int vbmf_b200_dense_upload(vbmf_b200_solver* s, const vbmf_b200_dense_state* st) {
    if (!s || !st) { set_error("NULL argument"); return -1; }
    if (check_dims(s, VBMF_B200_DENSE, st->L, st->M, st->H)) return -1;
    VB_CUDA_OK(cudaSetDevice(s->c->device));
    const Dev& d = s->d;
    const size_t HH = (size_t)d.H * d.H;
    if (up_A(s, st->AHat, nullptr) || up_B(s, st->BHat) || up(s, d.SigmaA, st->SigmaA, HH) || up(s, d.SigmaB, st->SigmaB, HH) ||
        up(s, d.CA, st->CA, HH) || up(s, d.CB, st->CB, HH) || up(s, d.invCA, st->invCA, HH) || up(s, d.invCB, st->invCB, HH)) return -1;
    memset(&s->h_sc, 0, sizeof(Scalars));
    s->h_sc.sigma2 = st->sigma2;
    s->h_sc.trYTY = s->c->trYTY;       // norm2(Y), src/vbmf.jl:154 (NaN while K0 still runs behind an asynchronous upload)
    if (push_scalars(s)) return -1;
    s->need_tr_copy = s->c->tr_pending;
    return 0;
}
extern "C" int vbmf_b200_dense_download(vbmf_b200_solver* s, vbmf_b200_dense_state* st) {
    if (!s || !st) { set_error("NULL argument"); return -1; }
    if (check_dims(s, VBMF_B200_DENSE, st->L, st->M, st->H)) return -1;
    VB_CUDA_OK(cudaSetDevice(s->c->device));
    const Dev& d = s->d;
    const size_t HH = (size_t)d.H * d.H;
    if (down_A(s, st->AHat, nullptr) || down_B(s, st->BHat) || down(s, st->SigmaA, d.SigmaA, HH) || down(s, st->SigmaB, d.SigmaB, HH) ||
        down(s, st->CA, d.CA, HH) || down(s, st->CB, d.CB, HH) || down(s, st->invCA, d.invCA, HH) || down(s, st->invCB, d.invCB, HH)) return -1;
    if (pull_scalars(s)) return -1;
    st->sigma2 = s->h_sc.sigma2;
    return down_yhat(s, st->YHat);
}

template <class ST>
static int sparse_like_upload(vbmf_b200_solver* s, const ST* st) {
    const Dev& d = s->d;
    const size_t HH = (size_t)d.H * d.H, MH = (size_t)d.Mloc * d.H;
    if (up_A(s, st->AHat, st->ATVecHat) || up_B(s, st->BHat) || up(s, d.SigmaA, st->SigmaA, HH) || up(s, d.SigmaB, st->SigmaB, HH) ||
        up(s, d.sdiag, st->diagSigmaATVec, MH) || up(s, d.CAv, st->CA, MH) || up(s, d.beta, st->beta, MH) ||
        up(s, d.CBv, st->CB, (size_t)d.H) || up(s, d.deltav, st->delta, (size_t)d.H) ||
        up(s, d.sigmaVec, st->sigmaVecHat, (size_t)d.L) || up(s, d.etaVec, st->etaVec, (size_t)d.L) || up(s, d.zetaVec, st->zetaVec, (size_t)d.L)) return -1;
    if (d.blocks != nullptr && st->SigmaATVec_blocks != nullptr && up(s, d.blocks, st->SigmaATVec_blocks, MH * d.H)) return -1;
    Scalars& h = s->h_sc;
    memset(&h, 0, sizeof(Scalars));
    h.gamma0 = st->gamma0; h.delta0 = st->delta0; h.gamma = st->gamma;
    h.sigmaHat = st->sigmaHat; h.eta0 = st->eta0; h.zeta0 = st->zeta0; h.eta = st->eta; h.zeta = st->zeta;
    h.trYTY = st->trYTY;
    return 0;
}
template <class ST>
static int sparse_like_download(vbmf_b200_solver* s, ST* st) {
    const Dev& d = s->d;
    const size_t HH = (size_t)d.H * d.H, MH = (size_t)d.Mloc * d.H;
    if (down_A(s, st->AHat, st->ATVecHat) || down_B(s, st->BHat) || down(s, st->SigmaA, d.SigmaA, HH) || down(s, st->SigmaB, d.SigmaB, HH) ||
        down(s, st->diagSigmaATVec, d.sdiag, MH) || down(s, st->CA, d.CAv, MH) || down(s, st->beta, d.beta, MH) ||
        down(s, st->CB, d.CBv, (size_t)d.H) || down(s, st->delta, d.deltav, (size_t)d.H) ||
        down(s, st->sigmaVecHat, d.sigmaVec, (size_t)d.L) || down(s, st->etaVec, d.etaVec, (size_t)d.L) || down(s, st->zetaVec, d.zetaVec, (size_t)d.L)) return -1;
    if (d.blocks != nullptr && st->SigmaATVec_blocks != nullptr && down(s, st->SigmaATVec_blocks, d.blocks, MH * d.H)) return -1;
    if (pull_scalars(s)) return -1;
    const Scalars& h = s->h_sc;
    st->sigmaHat = h.sigmaHat; st->zeta = h.zeta; st->eta = h.eta;
    return 0;
}

extern "C" int vbmf_b200_sparse_upload(vbmf_b200_solver* s, const vbmf_b200_sparse_state* st) {
    if (!s || !st) { set_error("NULL argument"); return -1; }
    if (check_dims(s, VBMF_B200_SPARSE, st->L, st->M, st->H)) return -1;
    VB_CUDA_OK(cudaSetDevice(s->c->device));
    if (sparse_like_upload(s, st)) return -1;
    s->h_sc.alpha0p = st->alpha0; s->h_sc.beta0p = st->beta0; s->h_sc.alpha = st->alpha;
    return push_scalars(s);
}
extern "C" int vbmf_b200_sparse_download(vbmf_b200_solver* s, vbmf_b200_sparse_state* st) {
    if (!s || !st) { set_error("NULL argument"); return -1; }
    if (check_dims(s, VBMF_B200_SPARSE, st->L, st->M, st->H)) return -1;
    VB_CUDA_OK(cudaSetDevice(s->c->device));
    if (sparse_like_download(s, st)) return -1;
    return down_yhat(s, st->YHat);
}
extern "C" int vbmf_b200_dual_upload(vbmf_b200_solver* s, const vbmf_b200_dual_state* st) {
    if (!s || !st) { set_error("NULL argument"); return -1; }
    if (check_dims(s, VBMF_B200_DUAL, st->L, st->M, st->H)) return -1;
    if (st->H0 != s->d.H0) { set_error("state H0 does not match the solver"); return -1; }
    VB_CUDA_OK(cudaSetDevice(s->c->device));
    if (sparse_like_upload(s, st)) return -1;
    Scalars& h = s->h_sc;
    h.alpha00 = st->alpha00; h.beta00 = st->beta00; h.alpha01 = st->alpha01; h.beta01 = st->beta01;
    h.alpha_g0 = st->alpha0; h.alpha_g1 = st->alpha1;
    return push_scalars(s);
}
extern "C" int vbmf_b200_dual_download(vbmf_b200_solver* s, vbmf_b200_dual_state* st) {
    if (!s || !st) { set_error("NULL argument"); return -1; }
    if (check_dims(s, VBMF_B200_DUAL, st->L, st->M, st->H)) return -1;
    VB_CUDA_OK(cudaSetDevice(s->c->device));
    // the interleaved vectors land in st->CA / st->beta; split them on the host (src/vbmf_dual.jl:340-350 in reverse)
    std::vector<double> tmpCA, tmpBeta, tmpA;
    const Dev& d = s->d;
    const size_t MH = (size_t)d.Mloc * d.H;
    vbmf_b200_dual_state w = *st;
    if (w.CA == nullptr) { tmpCA.resize(MH); w.CA = tmpCA.data(); }
    if (w.beta == nullptr) { tmpBeta.resize(MH); w.beta = tmpBeta.data(); }
    if (w.AHat == nullptr && (st->A0Hat || st->A1Hat)) { tmpA.resize(MH); w.AHat = tmpA.data(); }
    if (sparse_like_download(s, &w)) return -1;
    st->sigmaHat = w.sigmaHat; st->zeta = w.zeta; st->eta = w.eta;
    const Scalars& h = s->h_sc;
    st->alpha00 = h.alpha00; st->beta00 = h.beta00; st->alpha01 = h.alpha01; st->beta01 = h.beta01;
    st->alpha0 = h.alpha_g0; st->alpha1 = h.alpha_g1;
    if (st->alpha) { st->alpha[0] = h.alpha_g0; st->alpha[1] = h.alpha_g1; }
    const size_t M = (size_t)d.Mloc, H = (size_t)d.H, H0 = (size_t)d.H0, H1 = (size_t)d.H1;
    for (size_t m = 0; m < M; ++m) {
        for (size_t hh = 0; hh < H; ++hh) {
            const bool g1 = hh >= H0;
            const size_t k = g1 ? m * H1 + (hh - H0) : m * H0 + hh;
            double* ca = g1 ? st->CA1 : st->CA0;
            double* be = g1 ? st->beta1 : st->beta0;
            if (ca) ca[k] = w.CA[m * H + hh];
            if (be) be[k] = w.beta[m * H + hh];
        }
    }
    if (st->A0Hat) memcpy(st->A0Hat, w.AHat, M * H0 * 8);               // AHat[:, 1:H0], src/vbmf_dual.jl:283
    if (st->A1Hat) memcpy(st->A1Hat, w.AHat + M * H0, M * H1 * 8);      // AHat[:, H0+1:end]
    return down_yhat(s, st->YHat);
}

extern "C" int vbmf_b200_trial_upload(vbmf_b200_solver* s, const vbmf_b200_trial_state* st) {
    if (!s || !st) { set_error("NULL argument"); return -1; }
    if (check_dims(s, VBMF_B200_TRIAL, st->L, st->M, st->H)) return -1;
    if (st->H0 != s->d.H0 || st->M0 != s->d.M0) { set_error("state H0 / M0 do not match the solver"); return -1; }
    VB_CUDA_OK(cudaSetDevice(s->c->device));
    if (sparse_like_upload(s, st)) return -1;
    Scalars& h = s->h_sc;
    h.alpha00 = st->alpha01; h.beta00 = st->beta01; h.alpha01 = st->alpha02; h.beta01 = st->beta02; h.alpha02 = st->alpha03; h.beta02 = st->beta03;
    h.alpha_g0 = st->alpha1; h.alpha_g1 = st->alpha2; h.alpha_g2 = st->alpha3;
    return push_scalars(s);
}
extern "C" int vbmf_b200_trial_download(vbmf_b200_solver* s, vbmf_b200_trial_state* st) {
    if (!s || !st) { set_error("NULL argument"); return -1; }
    if (check_dims(s, VBMF_B200_TRIAL, st->L, st->M, st->H)) return -1;
    VB_CUDA_OK(cudaSetDevice(s->c->device));
    std::vector<double> tmpCA, tmpBeta, tmpA;
    const Dev& d = s->d;
    const size_t MH = (size_t)d.Mloc * d.H;
    vbmf_b200_trial_state w = *st;
    if (w.CA == nullptr) { tmpCA.resize(MH); w.CA = tmpCA.data(); }
    if (w.beta == nullptr) { tmpBeta.resize(MH); w.beta = tmpBeta.data(); }
    if (w.AHat == nullptr && (st->A1Hat || st->A2Hat || st->A3Hat)) { tmpA.resize(MH); w.AHat = tmpA.data(); }
    if (sparse_like_download(s, &w)) return -1;
    st->sigmaHat = w.sigmaHat; st->zeta = w.zeta; st->eta = w.eta;
    const Scalars& h = s->h_sc;
    st->alpha01 = h.alpha00; st->beta01 = h.beta00; st->alpha02 = h.alpha01; st->beta02 = h.beta01; st->alpha03 = h.alpha02; st->beta03 = h.beta02;
    st->alpha1 = h.alpha_g0; st->alpha2 = h.alpha_g1; st->alpha3 = h.alpha_g2;
    if (st->alpha) { st->alpha[0] = h.alpha_g0; st->alpha[1] = h.alpha_g1; st->alpha[2] = h.alpha_g2; }
    // split the interleaved vectors / AHat into the three groups (src/vbmf_trial.jl:316-319, 383-399 in reverse)
    const size_t M = (size_t)d.Mloc, H = (size_t)d.H, H0 = (size_t)d.H0, H1 = (size_t)d.H1;
    const long long m0loc = std::min<long long>(std::max<long long>((long long)d.M0 - d.moff, 0), (long long)M);   // local rows in group 2
    const size_t M2 = (size_t)m0loc, M3 = M - M2;
    for (size_t m = 0; m < M; ++m) {
        for (size_t hh = 0; hh < H; ++hh) {
            const double ca = w.CA[m * H + hh], be = w.beta[m * H + hh];
            if (hh < H0) { if (st->CA1) st->CA1[m * H0 + hh] = ca; if (st->beta1) st->beta1[m * H0 + hh] = be; }
            else if (m < M2) { const size_t k = m * H1 + (hh - H0); if (st->CA2) st->CA2[k] = ca; if (st->beta2) st->beta2[k] = be; }
            else { const size_t k = (m - M2) * H1 + (hh - H0); if (st->CA3) st->CA3[k] = ca; if (st->beta3) st->beta3[k] = be; }
        }
    }
    if (st->A1Hat) memcpy(st->A1Hat, w.AHat, M * H0 * 8);
    for (size_t hh = H0; hh < H; ++hh) {
        const double* colp = w.AHat + hh * M;
        if (st->A2Hat) memcpy(st->A2Hat + (hh - H0) * M2, colp, M2 * 8);
        if (st->A3Hat) memcpy(st->A3Hat + (hh - H0) * M3, colp + M2, M3 * 8);
    }
    return down_yhat(s, st->YHat);
}

// ---- enqueue helpers ---------------------------------------------------------------------------------------------------
// main stream after the (possibly still running) upload of Y and K0; the dense state's sum(Y.^2) follows device-side
static int settle_upload(vbmf_b200_solver* s) {
    if (ctx_wait_upload(s->c)) return -1;
    if (s->need_tr_copy) {
        if (k_copy_trYTY(s->c->st, s->d, s->c->d_tr)) return -1;
        s->need_tr_copy = false;
    }
    return 0;
}
static int enq_k1(vbmf_b200_solver* s, bool scaledB, bool reduce_slabs = true) {
    vbmf_b200_ctx* c = s->c;
    const Dev& d = s->d;
    if (c->Y == nullptr) { set_error("this step contracts with Y: attach Y first (the context only holds its shape)"); return -1; }
    if (settle_upload(s)) return -1;
    bool i8 = false;
    if (s->i8 && ctx_slices(c, &i8)) return -1;
    prof_mark(c, c->ev_k1);
    int rc;
    if (i8) {
        const size_t MH = (size_t)d.Mloc * d.H;
        rc = i8_k1(c, &s->i8o, scaledB ? d.Bs : d.B, d.ldB, d.H, s->S1 > 1 ? s->Ppart : d.P, s->S1, s->kbs1, d.sc);
        if (!rc && s->S1 > 1 && reduce_slabs) rc = k_sum_slabs(c->st, s->Ppart, s->S1, MH, d.P, d.sc);
    } else if (c->simt) rc = launch_gemm_ytb_simt(c->st, d.Y, d.ldY, scaledB ? d.Bs : d.B, d.ldB, d.P, d.Mloc, d.L, d.H, d.H, d.sc);
    else {
        const size_t MH = (size_t)d.Mloc * d.H;
        rc = launch_gemm_ytb(c->st, &c->tmY1, scaledB ? &s->tmBs : &s->tmB, s->S1 > 1 ? s->Ppart : d.P, d.Mloc, d.L, d.H, d.H,
                             s->S1, s->kbs1, MH, d.sc, c->num_sms);
        if (!rc && s->S1 > 1 && reduce_slabs) rc = k_sum_slabs(c->st, s->Ppart, s->S1, MH, d.P, d.sc);
    }
    prof_mark(c, c->ev_k1);
    prof_seg(c, SEG_K1);
    return rc;
}
static int enq_k2(vbmf_b200_solver* s) {
    vbmf_b200_ctx* c = s->c;
    const Dev& d = s->d;
    if (c->Y == nullptr) { set_error("this step contracts with Y: attach Y first (the context only holds its shape)"); return -1; }
    if (settle_upload(s)) return -1;
    bool i8 = false;
    if (s->i8 && ctx_slices(c, &i8)) return -1;
    prof_mark(c, c->ev_k2);
    int rc;
    if (i8) rc = i8_k2(c, &s->i8o, d.A, d.H, s->Qpart, d.ldB, s->S, s->kchunk, d.sc);
    else if (s->k2_simt) rc = launch_gemm_ya_simt(c->st, d.Y, d.ldY, d.A, s->Qpart, d.L, d.Mloc, d.H, d.ldB, s->kchunk, s->S, d.sc);
    else rc = launch_gemm_ya(c->st, &c->tmY2, &s->tmA, s->Qpart, d.L, d.Mloc, d.H, d.ldB, s->kchunk, s->S, d.sc, c->num_sms);
    prof_mark(c, c->ev_k2);
    prof_seg(c, SEG_K2);
    if (rc) return rc;
    rc = k_reduce_q(c->st, d, s->Qpart, s->S);
    prof_seg(c, SEG_REDUCE_Q);
    return rc;
}
// Grams of the current BHat that the A update / CB / sigma need
static int enq_gram_B(vbmf_b200_solver* s, int flags) {
    const Dev& d = s->d;
    cudaStream_t st = s->c->st;
    if (k_gram(st, d, d.B, false, d.L, nullptr, d.BtB)) return -1;
    if (d.kind != KIND_DENSE && (flags & F_DIAG_VAR)) {
        if (!s->mean_valid) { if (k_mean_sigma(st, d)) return -1; s->mean_valid = true; }
        if (flags & F_FULL_COV) { if (k_gram(st, d, d.B, false, d.L, d.sigmaVec, d.BtBw)) return -1; }   // B'diag(sv)B, src/vbmf_sparse.jl:182
        else { if (k_gram_w2(st, d, d.B, d.L, d.sigmaVec, d.BtBw)) return -1; }                            // norm2(B[:,h].*sv), :211 (Q4)
        if (k_scale_B(st, d)) return -1;
    }
    s->btb_valid = true;
    return 0;
}
static int copy_sa(vbmf_b200_solver* s) {   // step-level: SigmaA <- all-reduced sum of blocks right away
    const Dev& d = s->d;
    if (ctx_allreduce(s->c, d.packed + packed_sa(d), (size_t)d.H * d.H)) return -1;
    VB_CUDA_OK(cudaMemcpyAsync(d.SigmaA, d.packed + packed_sa(d), (size_t)d.H * d.H * 8, cudaMemcpyDeviceToDevice, s->c->st));
    return 0;
}
// main stream waits for the side-stream tail (post) of the previous iteration
static int wait_post(vbmf_b200_solver* s) {
    if (s->post_pending) {
        VB_CUDA_OK(cudaStreamWaitEvent(s->c->st, s->ev_p, 0));
        s->post_pending = false;
    }
    return 0;
}
static int enq_updateA(vbmf_b200_solver* s, int flags, bool fused) {
    const Dev& d = s->d;
    cudaStream_t st = s->c->st;
    if (!s->btb_valid) { if (wait_post(s) || enq_gram_B(s, flags)) return -1; }
    if (d.kind == KIND_DENSE) {
        // the epilogue sums the K1 slabs itself, multiplies by SigmaA/sigma2, masks, and leaves the local AHat'AHat in packed
        // K1 needs BHat only; everything after it needs the previous iteration's sigma2 / invCA (post) -> wait there
        // SigmaA needs B'B, SigmaB, sigma2 and inv(CA) only -- all final once the previous iteration's tail has run -- so inside
        // the loop it is inverted on the side stream right behind that tail, concurrently with K1 (enq_iteration)
        if (enq_k1(s, false, false) || wait_post(s)) return -1;
        if (!s->sigmaA_ahead && k_dense_sigmaA(st, d)) return -1;
        s->sigmaA_ahead = false;
        const bool slabs = !s->c->simt && s->S1 > 1;
        if (fused && (s->px || s->c->world == 1) && d.Mloc > 0) {
            // whole-loop run: the fixed-order sum of the Gram partials is only needed by SigmaB -> side stream (enq_updateB)
            if (k_dense_A_fused_range(st, d, slabs ? s->Ppart : d.P, slabs ? s->S1 : 1, (size_t)d.Mloc * d.H, 0, d.Mloc, 0, 1 << 30, &s->ata_parts)) return -1;
        } else if (k_dense_A_fused(st, d, slabs ? s->Ppart : d.P, slabs ? s->S1 : 1, (size_t)d.Mloc * d.H)) return -1;
        s->ata_local = true;
    } else {
        const bool dv = (flags & F_DIAG_VAR) != 0;
        // (H > 64: the fused kernel's 68 Gram accumulator registers leave one CTA per SM and it loses to the separate
        //  passes, 0.74 vs 0.55 ms at 125000 x 128)
        if (fused && !(flags & F_FULL_COV) && d.H <= 64) {
            // whole-loop diagonal path: slab sum, A, diag, mask, updateCA! and A'A in one pass over vec(A')
            if (enq_k1(s, dv, false) || wait_post(s)) return -1;
            const bool slabs = !s->c->simt && s->S1 > 1;
            // (the reduction of the partials is only needed by SigmaB and the tail: side stream, beside K2 -- enq_updateB)
            const bool defer = s->c->world == 1 || (s->px && !dv);
            if (k_sparse_A_diag_fused(st, d, slabs ? s->Ppart : d.P, slabs ? s->S1 : 1, (size_t)d.Mloc * d.H, flags, defer ? &s->diag_parts : nullptr)) return -1;
            s->ata_valid = false; s->q_valid = false;
            s->ata_local = true; s->ca_done = true;
            return 0;
        }
        if (enq_k1(s, dv) || wait_post(s)) return -1;
        if (flags & F_FULL_COV) { if (k_sparse_A_full(st, d, flags)) return -1; }
        else { if (k_sparse_A_diag(st, d, flags)) return -1; }
        if (k_mask(st, d)) return -1;
        if (!fused && copy_sa(s)) return -1;
    }
    s->ata_valid = false; s->q_valid = false;
    if (d.kind != KIND_DENSE) s->ata_local = false;
    s->ca_done = false;
    return 0;
}
static int enq_gram_A(vbmf_b200_solver* s) {
    const Dev& d = s->d;
    return k_gram(s->c->st, d, d.A, true, d.Mloc, nullptr, d.packed + packed_ata(d));
}
// Q = Y*AHat and AHat'AHat, all-reduced across shards.  fused: the payload also carries SigmaA blocks and dual sums.
static int enq_q_ata(vbmf_b200_solver* s, bool fused) {
    const Dev& d = s->d;
    if (!s->ata_local && enq_gram_A(s)) return -1;
    s->ata_local = false;
    if (enq_k2(s)) return -1;
    const size_t n = fused ? packed_len(d) : packed_sa(d);
    if (s->c->world > 1) prof_mark(s->c, s->c->ev_ar);
    if (ctx_allreduce(s->c, d.packed, n)) return -1;
    if (s->c->world > 1) prof_mark(s->c, s->c->ev_ar);
    s->ata_valid = true; s->q_valid = true;
    if (fused) s->extras_valid = true;
    return 0;
}
// the peers' regions of this solver as seen from this device; consumes `nbar` barrier epochs
static PxDev px_view(vbmf_b200_solver* s, int nbar, int site) {
    vbmf_b200_ctx* c = s->c;
    PxDev p;
    memset(&p, 0, sizeof(p));
    p.site = site;
    p.wait_ns = c->profile_segments ? c->px.wait_ns : nullptr;
    p.rank = c->rank; p.W = c->world; p.epoch = c->px.epoch;
    c->px.epoch += (unsigned long long)nbar;
    for (int r = 0; r < c->world; ++r) {
        char* base = r == c->rank ? c->px.local : c->px.peer[r];
        p.flags[r] = (unsigned long long*)base;
        p.packed[r] = (double*)(base + s->px_packed);
        p.B[r] = (double*)(base + s->px_B);
        p.gpart[r] = (double*)(base + s->px_gpart);
        p.small[r] = (double*)(base + s->px_small);
    }
    return p;
}
static int enq_updateB(vbmf_b200_solver* s, int flags, bool fused) {
    const Dev& d = s->d;
    cudaStream_t st = s->c->st;
    const bool px = fused && s->px && !(d.kind != KIND_DENSE && (flags & F_DIAG_VAR));
    if (px || (fused && s->c->world == 1)) {
        // px: updateB! with the exchange done by our own kernels over NVLink: the small sums are gathered from the peers, SigmaB
        // is inverted redundantly, every rank reduces its share of the rows of Y*AHat over the peers, runs the epilogue on
        // them and writes the new BHat rows to every peer; the Grams of BHat / BHat - Bold are exchanged as rank partials.
        // (The heteroscedastic row update needs all rows of the reduced Y*AHat on every rank: that case keeps the all-reduce.)
        // One GPU: nothing to exchange.  Either way SigmaB needs the A side of the iteration only, so the Gram partial sum,
        // the small exchange and the inverse run on the side stream beside K2 (their few CTAs share the SMs with K2's).
        if (d.kind != KIND_DENSE && (flags & F_DIAG_VAR) && !s->mean_valid) { if (k_mean_sigma(st, d)) return -1; s->mean_valid = true; }
        VB_CUDA_OK(cudaEventRecord(s->ev_a, st));
        VB_CUDA_OK(cudaStreamWaitEvent(s->side, s->ev_a, 0));
        // AHat'AHat (full covariance path: a Gram pass over AHat; otherwise the deferred sums of the A-side partials)
        if (!s->ata_local && k_gram(s->side, d, d.A, true, d.Mloc, nullptr, d.packed + packed_ata(d))) return -1;
        s->ata_local = false;
        if (s->ata_parts > 0 && k_sum_gram_partials(s->side, d, s->ata_parts)) return -1;
        s->ata_parts = 0;
        if (s->diag_parts > 0 && k_sparse_diag_reduce(s->side, d, s->diag_parts)) return -1;
        s->diag_parts = 0;
        if (px && k_px_small(s->side, d, px_view(s, 1, 0))) return -1;
        if (k_sigmaB(s->side, d, flags)) return -1;
        VB_CUDA_OK(cudaEventRecord(s->ev_sb, s->side));
        if (enq_k2(s)) return -1;
        if (px) prof_mark(s->c, s->c->ev_ar);
        VB_CUDA_OK(cudaStreamWaitEvent(st, s->ev_sb, 0));
        prof_seg(s->c, SEG_SIGMA_B);
        if (px) {
            int nparts = 1;
            if (k_B_epilogue_px(st, d, flags, px_view(s, 1, 1), &nparts)) return -1;
            prof_seg(s->c, SEG_B_EPI);
            if (k_B_reduce_px(st, d, px_view(s, 1, 2), nparts)) return -1;
            prof_seg(s->c, SEG_B_REDUCE);
            prof_mark(s->c, s->c->ev_ar);
        } else {
            if (k_B_epilogue(st, d, flags)) return -1;
            prof_seg(s->c, SEG_B_EPI);
        }
        s->ata_valid = true; s->extras_valid = true;
        s->q_valid = !px;                           // px: packed.Q is reduced on this rank's rows only
        s->btb_valid = !(d.kind != KIND_DENSE && (flags & F_DIAG_VAR));           // weighted Grams / Bs still stale with diag_var
        return 0;
    }
    if (!fused && d.kind != KIND_DENSE) {
        // step-level: packed.SA must hold the (global) SigmaA the state carries
        VB_CUDA_OK(cudaMemcpyAsync(d.packed + packed_sa(d), d.SigmaA, (size_t)d.H * d.H * 8, cudaMemcpyDeviceToDevice, st));
    }
    if (d.kind != KIND_DENSE && (flags & F_DIAG_VAR) && !s->mean_valid) { if (k_mean_sigma(st, d)) return -1; s->mean_valid = true; }
    if (enq_q_ata(s, fused)) return -1;
    prof_seg(s->c, SEG_EXCHANGE);
    if (k_sigmaB(st, d, flags)) return -1;
    prof_seg(s->c, SEG_SIGMA_B);
    if (k_B_epilogue(st, d, flags)) return -1;     // also BtB, DtD, tr(B'Q) of the new BHat
    prof_seg(s->c, SEG_B_EPI);
    s->btb_valid = !(d.kind != KIND_DENSE && (flags & F_DIAG_VAR));           // weighted Grams / Bs still stale with diag_var
    return 0;
}
static int enq_updateCA(vbmf_b200_solver* s, int flags, bool fused) {
    const Dev& d = s->d;
    if (d.kind == KIND_DENSE) {
        if (!s->ata_valid) {
            if (!s->ata_local && enq_gram_A(s)) return -1;
            s->ata_local = false;
            if (ctx_allreduce(s->c, d.packed + packed_ata(d), (size_t)d.H * d.H)) return -1;
            s->ata_valid = true;
        }
        return k_dense_cov_only(s->c->st, d, 0);
    }
    if (k_update_CA(s->c->st, d)) return -1;
    if ((d.kind == KIND_DUAL || d.kind == KIND_TRIAL) && !fused) { if (ctx_allreduce(s->c, d.packed + packed_ex(d), 8)) return -1; s->extras_valid = true; }
    return 0;
}

extern "C" int vbmf_b200_solver_step(vbmf_b200_solver* s, int step, int flags) {
    if (!s) { set_error("NULL solver"); return -1; }
    VB_CUDA_OK(cudaSetDevice(s->c->device));
    const Dev& d = s->d;
    cudaStream_t st = s->c->st;
    if (k_set_control(st, d, 1, 0.0, 0, 1)) return -1;
    int rc = 0;
    switch (step) {
        case VBMF_B200_STEP_UPDATE_A: rc = enq_updateA(s, flags, false); break;
        case VBMF_B200_STEP_UPDATE_B: rc = enq_updateB(s, flags, false); break;
        case VBMF_B200_STEP_UPDATE_CA: rc = enq_updateCA(s, flags, false); break;
        case VBMF_B200_STEP_UPDATE_CB:
            if (!s->btb_valid) rc = enq_gram_B(s, flags);
            if (!rc) rc = (d.kind == KIND_DENSE) ? k_dense_cov_only(st, d, 1) : k_updateCB_only(st, d);
            break;
        case VBMF_B200_STEP_UPDATE_SIGMA:
            if (!s->btb_valid) rc = enq_gram_B(s, flags);
            if (!rc && !s->q_valid) rc = enq_q_ata(s, false);
            if (!rc) rc = k_trbq(st, d);
            if (!rc) {
                if (d.kind != KIND_DENSE && (flags & F_DIAG_VAR)) { rc = k_sigma_rows(st, d); s->mean_valid = true; s->btb_valid = false; }
                else rc = k_sigma_only(st, d, flags);
            }
            break;
        case VBMF_B200_STEP_UPDATE_ALPHA00: case VBMF_B200_STEP_UPDATE_ALPHA01: case VBMF_B200_STEP_UPDATE_ALPHA02:
        case VBMF_B200_STEP_UPDATE_BETA00: case VBMF_B200_STEP_UPDATE_BETA01: case VBMF_B200_STEP_UPDATE_BETA02:
            if (d.kind != KIND_DUAL && d.kind != KIND_TRIAL) { set_error("hyper-prior steps exist for vbmf_dual / vbmf_trial only"); return -1; }
            if (d.kind == KIND_DUAL && (step == VBMF_B200_STEP_UPDATE_ALPHA02 || step == VBMF_B200_STEP_UPDATE_BETA02)) { set_error("vbmf_dual has two ARD groups"); return -1; }
            if (!s->extras_valid) {     // sum(CA_g), sum(log(beta_g)) of the CURRENT vectors; CA / beta stay as uploaded
                rc = k_update_CA(st, d, 1);
                if (!rc) rc = ctx_allreduce(s->c, d.packed + packed_ex(d), 8);
                s->extras_valid = true;
            }
            if (!rc) {
                int which = 0;      // 0..2 alpha of group 0..2, 3..5 beta of group 0..2
                switch (step) {
                    case VBMF_B200_STEP_UPDATE_ALPHA00: which = 0; break; case VBMF_B200_STEP_UPDATE_ALPHA01: which = 1; break;
                    case VBMF_B200_STEP_UPDATE_ALPHA02: which = 2; break; case VBMF_B200_STEP_UPDATE_BETA00: which = 3; break;
                    case VBMF_B200_STEP_UPDATE_BETA01: which = 4; break; default: which = 5; break;
                }
                rc = k_prior_only(st, d, which);
            }
            break;
        default: set_error("unknown step %d", step); return -1;
    }
    if (rc) return -1;
    VB_CUDA_OK(cudaStreamSynchronize(st));
    return 0;
}

static int enq_iteration(vbmf_b200_solver* s, int flags) {
    const Dev& d = s->d;
    cudaStream_t st = s->c->st;
    prof_seg(s->c, SEG_START);
    if (enq_updateA(s, flags, true)) return -1;                       // updateA!
    if (d.kind != KIND_DENSE && !s->ca_done && enq_updateCA(s, flags, true)) return -1;   // updateCA! (local; hoisted before the all-reduce)
    s->ca_done = false;
    prof_seg(s->c, SEG_A_EPI);
    if (enq_updateB(s, flags, true)) return -1;                       // updateB! (+ Grams of BHat and of BHat - Bold)
    if (d.kind != KIND_DENSE && (flags & F_DIAG_VAR)) {
        if (k_sigma_rows(st, d)) return -1;                           // updateSigma! (per-row)
        if (flags & F_FULL_COV) { if (k_gram(st, d, d.B, false, d.L, d.sigmaVec, d.BtBw)) return -1; }
        else { if (k_gram_w2(st, d, d.B, d.L, d.sigmaVec, d.BtBw)) return -1; }
        if (k_scale_B(st, d)) return -1;
    }
    s->btb_valid = true;
    // updateCA!/CB! (dense), updateCB!, updateSigma*!, priors, delta + loop control: on the side stream
    VB_CUDA_OK(cudaEventRecord(s->ev_b, st));
    VB_CUDA_OK(cudaStreamWaitEvent(s->side, s->ev_b, 0));
    if (k_post(s->side, d, flags, true)) return -1;
    if (d.kind == KIND_DENSE && s->loop_ahead) {       // SigmaA of the next iteration (skipped with it if the loop has just ended)
        if (k_dense_sigmaA(s->side, d)) return -1;
        s->sigmaA_ahead = true;
    }
    VB_CUDA_OK(cudaEventRecord(s->ev_p, s->side));
    s->post_pending = true;
    return 0;
}

// First dense iteration while Y is still arriving (asynchronous chunked attach): row m of AHat needs only column m of Y, and
// Y*AHat is a sum over columns, so updateA! and the Y*AHat part of updateB! run chunk by chunk behind the copy stream
// (K1, A epilogue, K2 and the slab reduction per chunk); the chunk results are summed in fixed order and the rest of the
// iteration (all-reduce, SigmaB, BHat epilogue, tail) is the usual one.  Every later iteration needs all of Y.
static int enq_iteration_chunked(vbmf_b200_solver* s, int flags) {
    vbmf_b200_ctx* c = s->c;
    const Dev& d = s->d;
    cudaStream_t st = c->st;
    const size_t nch = c->chunk_c0.size(), LH = (size_t)d.H * d.ldB, MH = (size_t)d.Mloc * d.H;
    if (s->Qc == nullptr || s->Qc_chunks < nch) {
        if (s->Qc) { VB_CUDA_OK(cudaStreamSynchronize(st)); cudaFree(s->Qc); s->Qc = nullptr; }
        if (cudaMalloc(&s->Qc, nch * LH * 8) != cudaSuccess) { cudaGetLastError(); set_error("cudaMalloc of the per-chunk Y*AHat buffer failed"); return -1; }
        s->Qc_chunks = nch;
    }
    if (!s->btb_valid) { if (wait_post(s) || enq_gram_B(s, flags)) return -1; }
    if (wait_post(s) || k_dense_sigmaA(st, d)) return -1;
    const bool slabs = s->S1 > 1;
    const int max_parts = std::max(1, (int)(MAX_PARTS / nch));
    int parts = 0;
    for (size_t k = 0; k < nch; ++k) {
        const int c0 = c->chunk_c0[k], n = c->chunk_n[k];
        VB_CUDA_OK(cudaStreamWaitEvent(st, c->ev_chunk[k], 0));
        CUtensorMap tmY1c, tmY2c, tmAc;
        const double* Yc = c->Y + (size_t)c0 * c->ldY;
        if (make_tmap_2d(&tmY1c, Yc, (uint64_t)c->L, (uint64_t)n, (uint64_t)c->ldY * 8, 16, 128)) return -1;
        if (make_tmap_2d(&tmY2c, Yc, (uint64_t)c->L, (uint64_t)n, (uint64_t)c->ldY * 8, 16, 16)) return -1;
        if (make_tmap_2d(&tmAc, d.A + (size_t)c0 * d.H, (uint64_t)d.H, (uint64_t)n, (uint64_t)d.H * 8, 16, 16)) return -1;
        // updateA! on the chunk: P = Y_c' * BHat (slabs at the chunk's rows), then the A epilogue on those rows
        if (launch_gemm_ytb(st, &tmY1c, &s->tmB, (slabs ? s->Ppart : d.P) + (size_t)c0 * d.H, n, d.L, d.H, d.H, s->S1, s->kbs1, MH, d.sc, c->num_sms)) return -1;
        int np = 0;
        if (k_dense_A_fused_range(st, d, slabs ? s->Ppart : d.P, slabs ? s->S1 : 1, MH, c0, c0 + n, parts, max_parts, &np)) return -1;
        parts += np;
        // Y_c * AHat_c -> Qc[k]
        int Sc = 1, kc = 16;
        plan_splitk(d.L, n, d.H, c->num_sms, &Sc, &kc);
        if (launch_gemm_ya(st, &tmY2c, &tmAc, s->Qpart, d.L, n, d.H, d.ldB, kc, Sc, d.sc, c->num_sms)) return -1;
        if (k_sum_slabs(st, s->Qpart, Sc, LH, s->Qc + k * LH, d.sc)) return -1;
    }
    c->chunks_pending = 0;                                   // the main stream is now ordered after every chunk
    if (k_sum_gram_partials(st, d, parts)) return -1;        // packed.AtA (local)
    if (k_sum_slabs(st, s->Qc, (int)nch, LH, d.packed + packed_q(d), d.sc)) return -1;
    s->ata_local = true;
    // sum(Y.^2) for updateSigma2!: K0 finishes on the statistics stream
    VB_CUDA_OK(cudaStreamWaitEvent(st, c->ev_stats, 0));
    if (s->need_tr_copy) { if (k_copy_trYTY(st, d, c->d_tr)) return -1; s->need_tr_copy = false; }
    // updateB! from the summed payload on
    if (ctx_allreduce(c, d.packed, packed_len(d))) return -1;
    s->ata_local = false; s->ata_valid = true; s->q_valid = true; s->extras_valid = true;
    if (k_sigmaB(st, d, flags) || k_B_epilogue(st, d, flags)) return -1;
    s->btb_valid = true;
    VB_CUDA_OK(cudaEventRecord(s->ev_b, st));
    VB_CUDA_OK(cudaStreamWaitEvent(s->side, s->ev_b, 0));
    if (k_post(s->side, d, flags, true)) return -1;
    VB_CUDA_OK(cudaEventRecord(s->ev_p, s->side));
    s->post_pending = true;
    return 0;
}

extern "C" int vbmf_b200_solver_run(vbmf_b200_solver* s, int64_t niter, double eps, int flags, int norm_mode,
                                    int64_t* iters, double* dout) {
    if (!s) { set_error("NULL solver"); return -1; }
    if (niter > 0x7fffffff) niter = 0x7fffffff;
    if (niter < 0) niter = 0;
    VB_CUDA_OK(cudaSetDevice(s->c->device));
    const Dev& d = s->d;
    cudaStream_t st = s->c->st;
    if (d.kind == KIND_DENSE) flags &= (F_EST_COVS | F_EST_VAR);
    if (k_set_control(st, d, (int)niter, eps, norm_mode, 0)) return -1;
    s->btb_valid = false;
    s->sigmaA_ahead = false;
    s->loop_ahead = true;
    if (enq_gram_B(s, flags) || k_norms_init(st, d)) return -1;      // old = BHat, src/vbmf.jl:188
    int64_t enq = 0;
    int slot = 0;
    bool pending = false;
    // Launch-bound regime (one iteration is ~12 launches of a few microseconds each): replay one captured iteration.
    const bool graph_mode = s->c->world == 1 && !s->px && !s->c->profile && niter >= 4 && getenv("VBMF_B200_NO_GRAPH") == nullptr &&
                            (double)d.L * (double)std::max(d.Mloc, 1) * (double)d.H < 4e9;
    if (graph_mode) {
        if (enq_iteration(s, flags) || wait_post(s)) return -1;       // first iteration eagerly (also settles one-time kernel attributes)
        enq = 1;
        if (s->gexec == nullptr || s->gexec_flags != flags) {
            if (s->gexec) { cudaGraphExecDestroy(s->gexec); s->gexec = nullptr; }
            cudaGraph_t graph = nullptr;
            VB_CUDA_OK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
            int rc = enq_iteration(s, flags);
            if (!rc) rc = wait_post(s);                              // joins the side stream back into the capture
            cudaError_t e = cudaStreamEndCapture(st, &graph);
            if (rc || e != cudaSuccess || graph == nullptr) { if (!rc) set_error("CUDA graph capture failed: %s", cudaGetErrorString(e)); cudaGetLastError(); return -1; }
            e = cudaGraphInstantiate(&s->gexec, graph, 0);
            cudaGraphDestroy(graph);
            if (e != cudaSuccess) { set_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(e)); s->gexec = nullptr; return -1; }
            s->gexec_flags = flags;
        }
        const int CHUNK_G = 8;
        while (enq < niter) {
            const int64_t c = std::min<int64_t>(CHUNK_G, niter - enq);
            for (int64_t i = 0; i < c; ++i) VB_CUDA_OK(cudaGraphLaunch(s->gexec, st));
            enq += c;
            VB_CUDA_OK(cudaMemcpyAsync(&s->h_flag[slot], &d.sc->active, sizeof(int), cudaMemcpyDeviceToHost, st));
            VB_CUDA_OK(cudaEventRecord(s->ev[slot], st));
            if (pending) {
                VB_CUDA_OK(cudaEventSynchronize(s->ev[slot ^ 1]));
                if (s->h_flag[slot ^ 1] == 0) break;
            }
            pending = true;
            slot ^= 1;
        }
    }
    // Y still arriving (asynchronous chunked attach) and the kind is dense: the first iteration follows the chunks
    if (!graph_mode && enq < niter && d.kind == KIND_DENSE && s->c->chunks_pending > 0 && !s->c->simt && !s->k2_simt && !s->c->profile &&
        s->c->Y != nullptr && getenv("VBMF_B200_NO_UPLOAD_OVERLAP") == nullptr) {
        if (enq_iteration_chunked(s, flags)) return -1;
        enq = 1;
    }
    const int CHUNK = 4;
    while (!graph_mode && enq < niter) {
        const int64_t c = std::min<int64_t>(CHUNK, niter - enq);
        for (int64_t i = 0; i < c; ++i) if (enq_iteration(s, flags)) return -1;
        enq += c;
        // the flag is produced on the side stream; copying it there keeps the main stream free of the dependency
        VB_CUDA_OK(cudaMemcpyAsync(&s->h_flag[slot], &d.sc->active, sizeof(int), cudaMemcpyDeviceToHost, s->side));
        VB_CUDA_OK(cudaEventRecord(s->ev[slot], s->side));
        if (pending) {
            VB_CUDA_OK(cudaEventSynchronize(s->ev[slot ^ 1]));
            if (s->h_flag[slot ^ 1] == 0) break;
        }
        pending = true;
        slot ^= 1;
    }
    s->loop_ahead = false; s->sigmaA_ahead = false;
    if (wait_post(s) || pull_scalars(s)) return -1;
    if (iters) *iters = s->h_sc.iter;
    if (dout) *dout = s->h_sc.d;
    if (s->h_sc.chol_fail & 4) {
        set_error("peer exchange: a rank did not reach a device-side barrier within ~30 s (did every rank enter the same call?); the state is invalid");
        return -1;
    }
    if (s->h_sc.chol_fail) { set_error("a posterior precision matrix was not positive definite (NaN written, loop ended)"); return -2; }
    return 0;
}

// The reference's loop with `update_log!(log, params)` after every iteration (src/vbmf.jl:206-208, src/vbmf_sparse.jl:385-387,
// src/vbmf_dual.jl:505-507): one device iteration at a time, the state stays resident, the callback downloads what it logs.
extern "C" int vbmf_b200_solver_run_logged(vbmf_b200_solver* s, int64_t niter, double eps, int flags, int norm_mode,
                                           vbmf_b200_iter_callback cb, void* user, int64_t* iters, double* dout) {
    if (!s) { set_error("NULL solver"); return -1; }
    int64_t done = 0;
    double d = eps + 1.0;                                   // src/vbmf.jl:189
    int rc = 0;
    while (done < niter && d > eps) {                       // while (i <= niter) && (d > eps)
        int64_t n = 0;
        rc = vbmf_b200_solver_run(s, 1, eps, flags, norm_mode, &n, &d);
        if (rc != 0 && rc != -2) return rc;
        if (n == 0) break;
        done += n;
        if (cb != nullptr && cb(user, s, done, d) != 0) break;   // non-zero return: stop early (the state stays valid)
        if (rc == -2) break;
    }
    if (iters) *iters = done;
    if (dout) *dout = d;
    return rc;
}

extern "C" int vbmf_b200_solver_lower_bound(vbmf_b200_solver* s, double trim, int trimmed, double* out) {
    if (!s || !out) { set_error("NULL argument"); return -1; }
    const Dev& d = s->d;
    if (d.kind == KIND_DENSE) { set_error("the dense solver has no lowerBound (the reference defines none)"); return -1; }
    VB_CUDA_OK(cudaSetDevice(s->c->device));
    cudaStream_t st = s->c->st;
    if (k_set_control(st, d, 1, 0.0, 0, 1)) return -1;
    if (enq_gram_B(s, 0)) return -1;
    if (!s->q_valid && enq_q_ata(s, false)) return -1;
    if (k_trbq(st, d)) return -1;
    if (k_lower_bound(st, d, trim, trimmed, 0)) return -1;
    if (ctx_allreduce(s->c, d.lbacc, 11)) return -1;
    if (k_lower_bound(st, d, trim, trimmed, 1)) return -1;
    if (pull_scalars(s)) return -1;
    *out = s->h_sc.lb;
    return 0;
}

extern "C" int vbmf_b200_solver_yhat(vbmf_b200_solver* s, double* YHat, int64_t ld) {
    if (!s || !YHat) { set_error("NULL argument"); return -1; }
    const Dev& d = s->d;
    VB_CUDA_OK(cudaSetDevice(s->c->device));
    if (d.Mloc == 0) return 0;
    double* tmp = nullptr;
    const size_t bytes = (size_t)d.L * d.Mloc * 8;
    if (cudaMalloc(&tmp, bytes) != cudaSuccess) { cudaGetLastError(); set_error("YHat needs %zu bytes of device memory", bytes); return -1; }
    int rc = k_yhat(s->c->st, d, tmp, d.L);
    if (!rc && cudaMemcpy2DAsync(YHat, (size_t)ld * 8, tmp, (size_t)d.L * 8, (size_t)d.L * 8, (size_t)d.Mloc, cudaMemcpyDeviceToHost, s->c->st) != cudaSuccess) { set_error("YHat download failed"); rc = -1; }
    cudaStreamSynchronize(s->c->st);
    cudaFree(tmp);
    return rc;
}

// ---- K1 / K2 on their own ------------------------------------------------------------------------------------------------
extern "C" int vbmf_b200_gemm_YtB(vbmf_b200_ctx* c, const double* B, int64_t H, double* P) {
    if (!c || !c->have_Y || !c->Y || !B || !P) { set_error("gemm_YtB: bad argument"); return -1; }
    if (H < 1 || H > 128) { set_error("H out of range"); return -1; }
    VB_CUDA_OK(cudaSetDevice(c->device));
    if (ctx_wait_upload(c)) return -1;
    const int ldB = (c->L + 1) & ~1;
    const size_t MH = (size_t)std::max(c->Mloc, 1) * H;
    double *dB = nullptr, *dP = nullptr, *dT = nullptr;
    VB_CUDA_OK(cudaMalloc(&dB, (size_t)H * ldB * 8));
    VB_CUDA_OK(cudaMalloc(&dP, MH * 8));
    VB_CUDA_OK(cudaMalloc(&dT, MH * 8));
    VB_CUDA_OK(cudaMemsetAsync(dB, 0, (size_t)H * ldB * 8, c->st));
    VB_CUDA_OK(cudaMemcpy2DAsync(dB, (size_t)ldB * 8, B, (size_t)c->L * 8, (size_t)c->L * 8, (size_t)H, cudaMemcpyHostToDevice, c->st));
    int rc = 0;
    bool i8 = false;
    I8Operands o;
    int S1 = 1, kbs1 = 1, S2 = 1, kc2 = 32;
    if (ctx_int8_wanted(c, H)) {
        i8_plans(c->L, c->Mloc, (int)H, c->num_sms, &S1, &kbs1, &S2, &kc2);
        rc = ctx_slices(c, &i8);
        if (!rc && i8) rc = i8_operands_alloc(&o, c->L, c->Mloc, (int)H, S2, &i8);
    }
    if (!rc && i8) {
        double* dPp = nullptr;
        if (S1 > 1 && cudaMalloc(&dPp, (size_t)S1 * MH * 8) != cudaSuccess) { set_error("cudaMalloc failed"); rc = -1; }
        if (!rc) rc = i8_k1(c, &o, dB, ldB, (int)H, S1 > 1 ? dPp : dP, S1, kbs1, nullptr);
        if (!rc && S1 > 1) rc = k_sum_slabs(c->st, dPp, S1, MH, dP, nullptr);
        if (dPp) { cudaStreamSynchronize(c->st); cudaFree(dPp); }
    } else if (!rc && c->simt) rc = launch_gemm_ytb_simt(c->st, c->Y, c->ldY, dB, ldB, dP, c->Mloc, c->L, (int)H, (int)H, nullptr);
    else if (!rc) {
        CUtensorMap tmB;
        rc = make_tmap_2d(&tmB, dB, (uint64_t)c->L, (uint64_t)H, (uint64_t)ldB * 8, 16, (uint32_t)gemm_geometry((int)H).bn);
        int S1 = 1, kbs1 = 1;
        plan_splitk_ytb(c->L, c->Mloc, (int)H, c->num_sms, &S1, &kbs1);
        double* dPp = nullptr;
        if (S1 > 1 && cudaMalloc(&dPp, (size_t)S1 * MH * 8) != cudaSuccess) { set_error("cudaMalloc failed"); rc = -1; }
        if (!rc) rc = launch_gemm_ytb(c->st, &c->tmY1, &tmB, S1 > 1 ? dPp : dP, c->Mloc, c->L, (int)H, (int)H, S1, kbs1, MH, nullptr, c->num_sms);
        if (!rc && S1 > 1) rc = k_sum_slabs(c->st, dPp, S1, MH, dP, nullptr);
        if (dPp) { cudaStreamSynchronize(c->st); cudaFree(dPp); }
    }
    if (!rc) rc = k_transpose(c->st, dP, dT, (int)H, c->Mloc);
    if (!rc && c->Mloc > 0 && cudaMemcpyAsync(P, dT, (size_t)c->Mloc * H * 8, cudaMemcpyDeviceToHost, c->st) != cudaSuccess) { set_error("copy failed"); rc = -1; }
    cudaError_t e = cudaStreamSynchronize(c->st);
    if (e != cudaSuccess) { set_error("gemm_YtB: %s", cudaGetErrorString(e)); rc = -1; }
    cudaFree(dB); cudaFree(dP); cudaFree(dT);
    return rc;
}

extern "C" int vbmf_b200_gemm_YA(vbmf_b200_ctx* c, const double* A, int64_t H, double* Q) {
    if (!c || !c->have_Y || !c->Y || !A || !Q) { set_error("gemm_YA: bad argument"); return -1; }
    if (H < 1 || H > 128) { set_error("H out of range"); return -1; }
    VB_CUDA_OK(cudaSetDevice(c->device));
    if (ctx_wait_upload(c)) return -1;
    const int ldQ = (c->L + 1) & ~1;
    const size_t MH = (size_t)std::max(c->Mloc, 1) * H;
    int S = 1, kchunk = 16;
    plan_splitk(c->L, c->Mloc, (int)H, c->num_sms, &S, &kchunk);
    bool i8 = false;
    I8Operands o;
    if (ctx_int8_wanted(c, H)) {
        int S1 = 1, kbs1 = 1;
        i8_plans(c->L, c->Mloc, (int)H, c->num_sms, &S1, &kbs1, &S, &kchunk);
        if (ctx_slices(c, &i8)) return -1;
        if (i8 && i8_operands_alloc(&o, c->L, c->Mloc, (int)H, S, &i8)) return -1;
    }
    double *dA = nullptr, *dT = nullptr, *dQp = nullptr, *dQ = nullptr;
    VB_CUDA_OK(cudaMalloc(&dA, MH * 8));
    VB_CUDA_OK(cudaMalloc(&dT, MH * 8));
    VB_CUDA_OK(cudaMalloc(&dQp, (size_t)S * H * ldQ * 8));
    VB_CUDA_OK(cudaMalloc(&dQ, (size_t)H * ldQ * 8));
    VB_CUDA_OK(cudaMemsetAsync(dQp, 0, (size_t)S * H * ldQ * 8, c->st));
    if (c->Mloc > 0) VB_CUDA_OK(cudaMemcpyAsync(dT, A, (size_t)c->Mloc * H * 8, cudaMemcpyHostToDevice, c->st));
    int rc = k_transpose(c->st, dT, dA, c->Mloc, (int)H);
    const bool simt = c->simt || (H % 2 != 0);
    if (!rc) {
        if (i8) rc = i8_k2(c, &o, dA, (int)H, dQp, ldQ, S, kchunk, nullptr);
        else if (simt) rc = launch_gemm_ya_simt(c->st, c->Y, c->ldY, dA, dQp, c->L, c->Mloc, (int)H, ldQ, kchunk, S, nullptr);
        else {
            CUtensorMap tmA;
            if (c->Mloc > 0) rc = make_tmap_2d(&tmA, dA, (uint64_t)H, (uint64_t)c->Mloc, (uint64_t)H * 8, 16, 16);
            if (!rc) rc = launch_gemm_ya(c->st, &c->tmY2, &tmA, dQp, c->L, c->Mloc, (int)H, ldQ, kchunk, S, nullptr, c->num_sms);
        }
    }
    if (!rc) {
        Dev d; memset(&d, 0, sizeof(d));
        d.H = (int)H; d.ldB = ldQ; d.L = c->L; d.packed = dQ;
        Scalars* none = nullptr; d.sc = none;
        // fixed-order slab reduction (same kernel as the solver path, unpredicated)
        rc = k_reduce_q(c->st, d, dQp, S);
    }
    if (!rc && cudaMemcpy2DAsync(Q, (size_t)c->L * 8, dQ, (size_t)ldQ * 8, (size_t)c->L * 8, (size_t)H, cudaMemcpyDeviceToHost, c->st) != cudaSuccess) { set_error("copy failed"); rc = -1; }
    cudaError_t e = cudaStreamSynchronize(c->st);
    if (e != cudaSuccess) { set_error("gemm_YA: %s", cudaGetErrorString(e)); rc = -1; }
    cudaFree(dA); cudaFree(dT); cudaFree(dQp); cudaFree(dQ);
    return rc;
}

// ---- one-call drop-ins ---------------------------------------------------------------------------------------------------
extern "C" int vbmf_b200_dense_run(vbmf_b200_ctx* c, vbmf_b200_dense_state* st, int64_t niter, double eps, int est_covs,
                                   int est_var, int norm_mode, int64_t* iters, double* d) {
    if (!c || !st) { set_error("NULL argument"); return -1; }
    vbmf_b200_solver* s = nullptr;
    if (vbmf_b200_solver_create(c, VBMF_B200_DENSE, st->H, st->H1, st->n_labels, st->labels, 0, &s)) return -1;
    int rc = vbmf_b200_dense_upload(s, st);
    if (!rc) rc = vbmf_b200_solver_run(s, niter, eps, (est_covs ? F_EST_COVS : 0) | (est_var ? F_EST_VAR : 0), norm_mode, iters, d);
    if (rc == 0 || rc == -2) { int r2 = vbmf_b200_dense_download(s, st); if (r2) rc = r2; }
    vbmf_b200_solver_destroy(s);
    return rc;
}
extern "C" int vbmf_b200_sparse_run(vbmf_b200_ctx* c, vbmf_b200_sparse_state* st, int64_t niter, double eps, int diag_var,
                                    int full_cov, int est_cb, int norm_mode, int64_t* iters, double* d) {
    if (!c || !st) { set_error("NULL argument"); return -1; }
    vbmf_b200_solver* s = nullptr;
    if (vbmf_b200_solver_create(c, VBMF_B200_SPARSE, st->H, st->H1, st->n_labels, st->labels, st->SigmaATVec_blocks != nullptr, &s)) return -1;
    int rc = vbmf_b200_sparse_upload(s, st);
    const int flags = (diag_var ? F_DIAG_VAR : 0) | (full_cov ? F_FULL_COV : 0) | (est_cb ? F_EST_CB : 0);
    if (!rc) rc = vbmf_b200_solver_run(s, niter, eps, flags, norm_mode, iters, d);
    if (rc == 0 || rc == -2) { int r2 = vbmf_b200_sparse_download(s, st); if (r2) rc = r2; }
    vbmf_b200_solver_destroy(s);
    return rc;
}
extern "C" int vbmf_b200_dual_run(vbmf_b200_ctx* c, vbmf_b200_dual_state* st, int64_t niter, double eps, int diag_var,
                                  int full_cov, int est_priors, int est_cb, int norm_mode, int64_t* iters, double* d) {
    if (!c || !st) { set_error("NULL argument"); return -1; }
    if (st->H < st->H0) { set_error("H must be at least H0!"); return -1; }
    vbmf_b200_solver* s = nullptr;
    if (vbmf_b200_solver_create(c, VBMF_B200_DUAL, st->H, st->H0, 0, nullptr, st->SigmaATVec_blocks != nullptr, &s)) return -1;
    int rc = vbmf_b200_dual_upload(s, st);
    const int flags = (diag_var ? F_DIAG_VAR : 0) | (full_cov ? F_FULL_COV : 0) | (est_cb ? F_EST_CB : 0) | (est_priors ? F_EST_PRIORS : 0);
    if (!rc) rc = vbmf_b200_solver_run(s, niter, eps, flags, norm_mode, iters, d);
    if (rc == 0 || rc == -2) { int r2 = vbmf_b200_dual_download(s, st); if (r2) rc = r2; }
    vbmf_b200_solver_destroy(s);
    return rc;
}

extern "C" int vbmf_b200_trial_run(vbmf_b200_ctx* c, vbmf_b200_trial_state* st, int64_t niter, double eps, int diag_var, int full_cov,
                                   int est_priors, int est_cb, int norm_mode, int64_t* iters, double* d) {
    if (!c || !st) { set_error("NULL argument"); return -1; }
    if (st->H < st->H0) { set_error("H must be at least H0!"); return -1; }
    vbmf_b200_solver* s = nullptr;
    if (vbmf_b200_solver_create_trial(c, st->H, st->H0, st->M0, st->SigmaATVec_blocks != nullptr, &s)) return -1;
    int rc = vbmf_b200_trial_upload(s, st);
    const int flags = (diag_var ? F_DIAG_VAR : 0) | (full_cov ? F_FULL_COV : 0) | (est_cb ? F_EST_CB : 0) | (est_priors ? F_EST_PRIORS : 0);
    if (!rc) rc = vbmf_b200_solver_run(s, niter, eps, flags, norm_mode, iters, d);
    if (rc == 0 || rc == -2) { int r2 = vbmf_b200_trial_download(s, st); if (r2) rc = r2; }
    vbmf_b200_solver_destroy(s);
    return rc;
}

// ---- K11: batched vbls! ----------------------------------------------------------------------------------------------------

// host-side packing / unpacking of many small problems: a few threads over disjoint problem ranges (plain memcpy work)
template <class F> static void parallel_for(int64_t n, F&& fn) {
    const unsigned hw = std::thread::hardware_concurrency();
    const int T = (int)std::min<int64_t>(std::min<unsigned>(hw ? hw : 1u, 8u), n / 64);
    if (T <= 1) { for (int64_t p = 0; p < n; ++p) fn(p); return; }
    std::vector<std::thread> th;
    th.reserve(T);
    for (int t = 0; t < T; ++t)
        th.emplace_back([&fn, n, t, T] { for (int64_t p = n * t / T; p < n * (t + 1) / T; ++p) fn(p); });
    for (auto& x : th) x.join();
}

// grow-only staging of the batched path: device arena + pinned host mirror with identical offsets
static int batch_reserve(vbmf_b200_ctx* c, size_t total) {
    if (total <= c->batch_bytes) return 0;
    VB_CUDA_OK(cudaStreamSynchronize(c->st));
    if (c->batch_dev) cudaFree(c->batch_dev);
    if (c->batch_host) cudaFreeHost(c->batch_host);
    c->batch_dev = c->batch_host = nullptr; c->batch_bytes = 0;
    const size_t cap = total + total / 4;
    if (cudaMalloc(&c->batch_dev, cap) != cudaSuccess || cudaHostAlloc(&c->batch_host, cap, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        if (c->batch_dev) { cudaFree(c->batch_dev); c->batch_dev = nullptr; }
        set_error("batched vbls: allocating %zu staging bytes failed", cap);
        return -1;
    }
    c->batch_bytes = cap;
    return 0;
}

// Routes every problem of a batch (batched_cluster_size) and orders them for the launches: plist = the one-CTA problems,
// then those of cluster size 1, 2, 4, 8; n[g] = count of group g; Mmax0 = largest M of the one-CTA problems.
static void batch_route(int kind, int L, int H, const std::vector<int>& moff, std::vector<int>& plist, int (&n)[5], int& Mmax0) {
    const int nprob = (int)moff.size() - 1;
    std::vector<int> grp(nprob);
    for (int g = 0; g < 5; ++g) n[g] = 0;
    Mmax0 = 0;
    for (int p = 0; p < nprob; ++p) {
        const int M = moff[p + 1] - moff[p], cs = vb::batched_cluster_size(kind, L, H, M);
        int g = 0;
        while (g < 4 && cs > (g == 0 ? 0 : 1 << (g - 1))) ++g;
        grp[p] = g;
        ++n[g];
        if (g == 0) Mmax0 = std::max(Mmax0, M);
    }
    plist.clear();
    for (int g = 0; g < 5; ++g) for (int p = 0; p < nprob; ++p) if (grp[p] == g) plist.push_back(p);
}

extern "C" int vbmf_b200_batched_plan(int kind, int64_t L, int64_t H, int full_cov, int diag_var, int64_t nprob, const int64_t* M,
                                      int32_t* cluster_out) {
    if (kind < VBMF_B200_DENSE || kind > VBMF_B200_TRIAL) { set_error("batched_plan: unknown parameter kind %d", kind); return -1; }
    const int64_t Hmax = kind == VBMF_B200_DENSE ? 32 : 64;
    if (H < 1 || H > Hmax) { set_error("batched vbls supports 1 <= H <= %lld (got H = %lld)", (long long)Hmax, (long long)H); return -1; }
    if (L < 1 || L > 0x7fffff00LL || nprob < 0 || (nprob > 0 && (!M || !cluster_out)) || (full_cov != 0 && full_cov != 1) ||
        (diag_var != 0 && diag_var != 1)) {
        set_error("batched_plan: bad argument"); return -1;
    }
    for (int64_t p = 0; p < nprob; ++p)
        if (M[p] < 1 || M[p] > 0x7fffff00LL) { set_error("batched_plan: bad argument (M of problem %lld)", (long long)p); return -1; }
    for (int64_t p = 0; p < nprob; ++p) cluster_out[p] = vb::batched_cluster_size(kind, (int)L, (int)H, (int)M[p]);
    return 0;
}

template <class ST> struct BatchView {
    static const ST* get(void* const* states, int64_t p) { return (const ST*)states[p]; }
};

template <class ST>
static int batched_vbls_impl(vbmf_b200_ctx* c, int kind, int64_t nprob, const double* const* Y, void* const* states,
                             int64_t niter, int flags) {
    if (nprob <= 0) return 0;
    const bool dvar = (flags & F_DIAG_VAR) != 0;
    const ST* s0 = (const ST*)states[0];
    const int64_t L = s0->L, H = s0->H;
    constexpr bool IS_DUAL = std::is_same<ST, vbmf_b200_dual_state>::value, IS_TRIAL = std::is_same<ST, vbmf_b200_trial_state>::value;
    int64_t H0 = H;
    if constexpr (IS_DUAL || IS_TRIAL) H0 = s0->H0;
    if (L < 1 || H < 1 || H > 64) { set_error("batched vbls supports 1 <= H <= 64 (got H = %lld)", (long long)H); return -1; }
    if (H0 < 0 || H0 > H) { set_error("H must be at least H0!"); return -1; }
    std::vector<int> moff(nprob + 1, 0);
    bool want_yhat = false, want_blocks = false;
    for (int64_t p = 0; p < nprob; ++p) {
        const ST* s = (const ST*)states[p];
        if (s == nullptr || Y[p] == nullptr) { set_error("batched vbls: NULL problem %lld", (long long)p); return -1; }
        if (s->L != L || s->H != H || s->M < 1) { set_error("batched vbls: problem %lld has different L/H or M < 1", (long long)p); return -1; }
        if constexpr (IS_DUAL || IS_TRIAL) { if (s->H0 != H0) { set_error("batched vbls: H0 differs"); return -1; } }
        else { if (s->n_labels > 0 && s->H1 > 0) { set_error("batched vbls: labels are not supported"); return -1; } }
        if (dvar && (s->sigmaVecHat == nullptr || s->etaVec == nullptr)) { set_error("batched vbls: diag_var needs sigmaVecHat / etaVec of problem %lld", (long long)p); return -1; }
        moff[p + 1] = moff[p] + (int)s->M;
        want_yhat = want_yhat || s->YHat != nullptr;
        want_blocks = want_blocks || s->SigmaATVec_blocks != nullptr;
    }
    const size_t Mtot = (size_t)moff[nprob], MH = Mtot * H, HH = (size_t)H * H, LH = (size_t)L * H;
    VB_CUDA_OK(cudaSetDevice(c->device));
    // ---- one arena, laid out [inputs | in-out | outputs]; the pinned host mirror uses the same offsets so the whole
    //      upload is one copy of [0, up_end) and the whole download one copy of [down_begin, total)
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += align_up(bytes, 256); return o; };
    std::vector<int> plist;
    int ngrp[5], Mmax0;
    batch_route(kind, (int)L, (int)H, moff, plist, ngrp, Mmax0);
    const bool wide = ngrp[0] < nprob;
    const size_t o_moff = take((size_t)(nprob + 1) * 4), o_pl = take((size_t)nprob * 4), o_Y = take(L * Mtot * 8), o_B = take(nprob * LH * 8),
                 o_SB = take(nprob * HH * 8);
    const size_t down_begin = off;
    const size_t o_CA = take(MH * 8), o_sc = take((size_t)nprob * 16 * 8);
    const size_t o_sv = dvar ? take((size_t)nprob * L * 8) : 0, o_ev = dvar ? take((size_t)nprob * L * 8) : 0;
    const size_t up_end = off;
    const size_t o_A = take(MH * 8), o_beta = take(MH * 8), o_s = take(MH * 8), o_SA = take(nprob * HH * 8);
    const size_t o_zv = dvar ? take((size_t)nprob * L * 8) : 0;
    const size_t o_YH = want_yhat ? take(L * Mtot * 8) : 0, o_blk = want_blocks ? take(MH * H * 8) : 0;
    const size_t total = off;
    // device-only working storage of the wide kernel, neither uploaded nor downloaded
    const size_t o_V = wide ? take(MH * 8) : 0, o_rv = wide && dvar ? take((size_t)nprob * (1 + BATCH_MAX_CLUSTER) * L * 8) : 0;
    if (batch_reserve(c, off)) return -1;
    char* hb = c->batch_host;
    char* db = c->batch_dev;
    // ---- pack
    memcpy(hb + o_moff, moff.data(), (size_t)(nprob + 1) * 4);
    memcpy(hb + o_pl, plist.data(), (size_t)nprob * 4);
    double *hY = (double*)(hb + o_Y), *hB = (double*)(hb + o_B), *hSB = (double*)(hb + o_SB), *hCA = (double*)(hb + o_CA), *hsc = (double*)(hb + o_sc);
    memset(hsc, 0, (size_t)nprob * 16 * 8);
    parallel_for(nprob, [&](int64_t p) {
        const ST* s = (const ST*)states[p];
        memcpy(&hY[(size_t)moff[p] * L], Y[p], (size_t)s->M * L * 8);
        memcpy(&hB[p * LH], s->BHat, LH * 8);
        memcpy(&hSB[p * HH], s->SigmaB, HH * 8);
        memcpy(&hCA[(size_t)moff[p] * H], s->CA, (size_t)s->M * H * 8);
        if (dvar) {
            memcpy((double*)(hb + o_sv) + (size_t)p * L, s->sigmaVecHat, (size_t)L * 8);
            memcpy((double*)(hb + o_ev) + (size_t)p * L, s->etaVec, (size_t)L * 8);
        }
        double* sc = &hsc[(size_t)p * 16];
        sc[0] = s->sigmaHat; sc[1] = s->eta; sc[2] = s->zeta; sc[3] = s->zeta0; sc[4] = s->trYTY;
        if constexpr (IS_DUAL) { sc[7] = s->alpha00; sc[8] = s->beta00; sc[9] = s->alpha01; sc[10] = s->beta01; }
        else if constexpr (IS_TRIAL) {
            sc[5] = (double)std::min<int64_t>(std::max<int64_t>(s->M0, 0), s->M);
            sc[7] = s->alpha01; sc[8] = s->beta01; sc[9] = s->alpha02; sc[10] = s->beta02; sc[14] = s->alpha03; sc[15] = s->beta03;
        } else { sc[5] = s->alpha; sc[6] = s->beta0; }
    });
    int rc = 0;
    cudaStream_t st = c->st;
    if (cudaMemcpyAsync(db, hb, up_end, cudaMemcpyHostToDevice, st) != cudaSuccess) { cudaGetLastError(); set_error("batched vbls: upload failed"); return -1; }
    BatchDesc bd;
    bd.nprob = (int)nprob; bd.L = (int)L; bd.H = (int)H; bd.H0 = (int)H0; bd.kind = kind; bd.niter = (int)std::max<int64_t>(niter, 0);
    bd.full_cov = (flags & F_FULL_COV) ? 1 : 0; bd.Mmax = Mmax0;
    bd.moff = (const int*)(db + o_moff); bd.Y = (const double*)(db + o_Y); bd.B = (const double*)(db + o_B); bd.SigmaB = (const double*)(db + o_SB);
    bd.A = (double*)(db + o_A); bd.CA = (double*)(db + o_CA); bd.beta = (double*)(db + o_beta); bd.sdiag = (double*)(db + o_s);
    bd.SigmaA = (double*)(db + o_SA); bd.blocks = want_blocks ? (double*)(db + o_blk) : nullptr; bd.YHat = want_yhat ? (double*)(db + o_YH) : nullptr;
    bd.scal = (double*)(db + o_sc);
    bd.diag_var = dvar ? 1 : 0;
    bd.sigmaVec = dvar ? (double*)(db + o_sv) : nullptr; bd.etaVec = dvar ? (const double*)(db + o_ev) : nullptr;
    bd.zetaVec = dvar ? (double*)(db + o_zv) : nullptr;
    bd.plist = (const int*)(db + o_pl);
    bd.V = wide ? (double*)(db + o_V) : nullptr;
    bd.rowv = wide && dvar ? (double*)(db + o_rv) : nullptr;
    prof_mark(c, c->ev_k1);       // profiling: the kernels alone (read back through vbmf_b200_ctx_profile_read, K1 slot)
    if (bd.niter > 0) rc = k_batched_vbls(st, bd, ngrp, Mmax0);
    prof_mark(c, c->ev_k1);
    // ---- download + unpack
    if (!rc && bd.niter > 0 && cudaMemcpyAsync(hb + down_begin, db + down_begin, total - down_begin, cudaMemcpyDeviceToHost, st) != cudaSuccess) {
        cudaGetLastError(); set_error("batched vbls: download failed"); rc = -1;
    }
    { cudaError_t e = cudaStreamSynchronize(st); if (e != cudaSuccess && !rc) { set_error("batched vbls: %s", cudaGetErrorString(e)); rc = -1; } }
    if (rc || bd.niter == 0) return rc;
    const double *hA = (const double*)(hb + o_A), *hbeta = (const double*)(hb + o_beta), *hs = (const double*)(hb + o_s), *hSA = (const double*)(hb + o_SA),
                 *hYH = (const double*)(hb + o_YH), *hblk = (const double*)(hb + o_blk);
    std::atomic<bool> failed(false);
    parallel_for(nprob, [&](int64_t p) {
        ST* s = (ST*)states[p];
        const size_t M = (size_t)s->M, o = (size_t)moff[p] * H;
        const double* sc = &hsc[(size_t)p * 16];
        if (sc[13] != 0.0) failed.store(true);
        if (s->ATVecHat) memcpy(s->ATVecHat, &hA[o], M * H * 8);
        if (s->AHat) for (size_t m = 0; m < M; ++m) for (size_t h = 0; h < (size_t)H; ++h) s->AHat[h * M + m] = hA[o + m * H + h];
        if (s->diagSigmaATVec) memcpy(s->diagSigmaATVec, &hs[o], M * H * 8);
        if (s->CA) memcpy(s->CA, &hCA[o], M * H * 8);
        if (s->beta) memcpy(s->beta, &hbeta[o], M * H * 8);
        if (s->SigmaA) memcpy(s->SigmaA, &hSA[p * HH], HH * 8);
        if (s->YHat) memcpy(s->YHat, &hYH[(size_t)moff[p] * L], M * L * 8);
        if (s->SigmaATVec_blocks) memcpy(s->SigmaATVec_blocks, &hblk[o * H], M * HH * 8);
        if (dvar) {
            if (s->sigmaVecHat) memcpy(s->sigmaVecHat, (const double*)(hb + o_sv) + (size_t)p * L, (size_t)L * 8);
            if (s->zetaVec) memcpy(s->zetaVec, (const double*)(hb + o_zv) + (size_t)p * L, (size_t)L * 8);
        }
        s->sigmaHat = sc[0]; s->zeta = sc[2];
        if constexpr (IS_TRIAL) {
            s->alpha1 = sc[11]; s->alpha2 = sc[12]; s->alpha3 = sc[6];
            if (s->alpha) { s->alpha[0] = sc[11]; s->alpha[1] = sc[12]; s->alpha[2] = sc[6]; }
            const size_t h0 = (size_t)H0, h1 = (size_t)(H - H0);
            const size_t M2 = (size_t)std::min<int64_t>(std::max<int64_t>(s->M0, 0), s->M), M3 = M - M2;
            for (size_t m = 0; m < M; ++m) for (size_t h = 0; h < (size_t)H; ++h) {
                const double ca = hCA[o + m * H + h], be = hbeta[o + m * H + h], av = hA[o + m * H + h];
                if (h < h0) {
                    if (s->CA1) s->CA1[m * h0 + h] = ca;
                    if (s->beta1) s->beta1[m * h0 + h] = be;
                    if (s->A1Hat) s->A1Hat[h * M + m] = av;
                } else if (m < M2) {
                    const size_t k = m * h1 + (h - h0);
                    if (s->CA2) s->CA2[k] = ca;
                    if (s->beta2) s->beta2[k] = be;
                    if (s->A2Hat) s->A2Hat[(h - h0) * M2 + m] = av;
                } else {
                    const size_t k = (m - M2) * h1 + (h - h0);
                    if (s->CA3) s->CA3[k] = ca;
                    if (s->beta3) s->beta3[k] = be;
                    if (s->A3Hat) s->A3Hat[(h - h0) * M3 + (m - M2)] = av;
                }
            }
        }
        if constexpr (IS_DUAL) {
            s->alpha0 = sc[11]; s->alpha1 = sc[12];
            if (s->alpha) { s->alpha[0] = sc[11]; s->alpha[1] = sc[12]; }
            const size_t h0 = (size_t)H0, h1 = (size_t)(H - H0);
            for (size_t m = 0; m < M; ++m) for (size_t h = 0; h < (size_t)H; ++h) {
                const bool g1 = h >= h0;
                const size_t k = g1 ? m * h1 + (h - h0) : m * h0 + h;
                if (g1) { if (s->CA1) s->CA1[k] = hCA[o + m * H + h]; if (s->beta1) s->beta1[k] = hbeta[o + m * H + h]; }
                else { if (s->CA0) s->CA0[k] = hCA[o + m * H + h]; if (s->beta0) s->beta0[k] = hbeta[o + m * H + h]; }
                if (g1) { if (s->A1Hat) s->A1Hat[(h - h0) * M + m] = hA[o + m * H + h]; }
                else { if (s->A0Hat) s->A0Hat[h * M + m] = hA[o + m * H + h]; }
            }
        }
    });
    if (failed.load()) { set_error("batched vbls: a per-column precision matrix was not positive definite (NaN written)"); return -2; }
    return 0;
}


// dense `vbmf_parameters` problems (class_alg = "vbls", examples/mil_util.jl:470-478)
static int batched_vbls_dense_impl(vbmf_b200_ctx* c, int64_t nprob, const double* const* Y, void* const* states, int64_t niter) {
    if (nprob <= 0) return 0;
    typedef vbmf_b200_dense_state ST;
    const ST* s0 = (const ST*)states[0];
    const int64_t L = s0->L, H = s0->H;
    if (L < 1 || H < 1 || H > 32) { set_error("batched vbls supports 1 <= H <= 32 (got H = %lld)", (long long)H); return -1; }
    std::vector<int> moff(nprob + 1, 0);
    bool want_yhat = false;
    for (int64_t p = 0; p < nprob; ++p) {
        const ST* s = (const ST*)states[p];
        if (s == nullptr || Y[p] == nullptr) { set_error("batched vbls: NULL problem %lld", (long long)p); return -1; }
        if (s->L != L || s->H != H || s->M < 1) { set_error("batched vbls: problem %lld has different L/H or M < 1", (long long)p); return -1; }
        if (s->n_labels > 0 && s->H1 > 0) { set_error("batched vbls: labels are not supported"); return -1; }
        for (int64_t a = 0; a < H; ++a) for (int64_t b = 0; b < H; ++b)
            if (a != b && s->invCA[a + b * H] != 0.0) { set_error("batched vbls: invCA of problem %lld is not diagonal", (long long)p); return -1; }
        moff[p + 1] = moff[p] + (int)s->M;
        want_yhat = want_yhat || s->YHat != nullptr;
    }
    const size_t Mtot = (size_t)moff[nprob], MH = Mtot * H, HH = (size_t)H * H, LH = (size_t)L * H;
    VB_CUDA_OK(cudaSetDevice(c->device));
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += align_up(bytes, 256); return o; };
    std::vector<int> plist;
    int ngrp[5], Mmax0;
    batch_route(VBMF_B200_DENSE, (int)L, (int)H, moff, plist, ngrp, Mmax0);
    const bool wide = ngrp[0] < nprob;
    const size_t o_moff = take((size_t)(nprob + 1) * 4), o_pl = take((size_t)nprob * 4), o_Y = take(L * Mtot * 8), o_B = take(nprob * LH * 8),
                 o_SB = take(nprob * HH * 8);
    const size_t down_begin = off;
    const size_t o_ic = take(nprob * H * 8), o_sc = take((size_t)nprob * 16 * 8);
    const size_t up_end = off;
    const size_t o_A = take(MH * 8), o_SA = take(nprob * HH * 8), o_c = take(nprob * H * 8);
    const size_t o_YH = want_yhat ? take(L * Mtot * 8) : 0;
    const size_t total = off;
    const size_t o_V = wide ? take(MH * 8) : 0;      // device-only working storage of the wide kernel
    if (batch_reserve(c, off)) return -1;
    char* hb = c->batch_host;
    char* db = c->batch_dev;
    memcpy(hb + o_moff, moff.data(), (size_t)(nprob + 1) * 4);
    memcpy(hb + o_pl, plist.data(), (size_t)nprob * 4);
    double *hY = (double*)(hb + o_Y), *hB = (double*)(hb + o_B), *hSB = (double*)(hb + o_SB), *hic = (double*)(hb + o_ic), *hsc = (double*)(hb + o_sc);
    memset(hsc, 0, (size_t)nprob * 16 * 8);
    for (int64_t p = 0; p < nprob; ++p) {
        const ST* s = (const ST*)states[p];
        memcpy(&hY[(size_t)moff[p] * L], Y[p], (size_t)s->M * L * 8);
        memcpy(&hB[p * LH], s->BHat, LH * 8);
        memcpy(&hSB[p * HH], s->SigmaB, HH * 8);
        for (int64_t h = 0; h < H; ++h) hic[p * H + h] = s->invCA[h + h * H];
        hsc[(size_t)p * 16] = s->sigma2;
    }
    cudaStream_t st = c->st;
    if (cudaMemcpyAsync(db, hb, up_end, cudaMemcpyHostToDevice, st) != cudaSuccess) { cudaGetLastError(); set_error("batched vbls: upload failed"); return -1; }
    BatchDenseDesc bd;
    bd.nprob = (int)nprob; bd.L = (int)L; bd.H = (int)H; bd.niter = (int)std::max<int64_t>(niter, 0); bd.Mmax = Mmax0;
    bd.moff = (const int*)(db + o_moff); bd.Y = (const double*)(db + o_Y); bd.B = (const double*)(db + o_B); bd.SigmaB = (const double*)(db + o_SB);
    bd.A = (double*)(db + o_A); bd.SigmaA = (double*)(db + o_SA); bd.icA = (double*)(db + o_ic); bd.cA = (double*)(db + o_c);
    bd.YHat = want_yhat ? (double*)(db + o_YH) : nullptr; bd.scal = (double*)(db + o_sc);
    bd.plist = (const int*)(db + o_pl); bd.V = wide ? (double*)(db + o_V) : nullptr;
    int rc = 0;
    prof_mark(c, c->ev_k1);
    if (bd.niter > 0) rc = k_batched_vbls_dense(st, bd, ngrp, Mmax0);
    prof_mark(c, c->ev_k1);
    if (!rc && bd.niter > 0 && cudaMemcpyAsync(hb + down_begin, db + down_begin, total - down_begin, cudaMemcpyDeviceToHost, st) != cudaSuccess) {
        cudaGetLastError(); set_error("batched vbls: download failed"); rc = -1;
    }
    { cudaError_t e = cudaStreamSynchronize(st); if (e != cudaSuccess && !rc) { set_error("batched vbls: %s", cudaGetErrorString(e)); rc = -1; } }
    if (rc || bd.niter == 0) return rc;
    const double *hA = (const double*)(hb + o_A), *hSA = (const double*)(hb + o_SA), *hc = (const double*)(hb + o_c), *hYH = (const double*)(hb + o_YH);
    bool failed = false;
    for (int64_t p = 0; p < nprob; ++p) {
        ST* s = (ST*)states[p];
        const size_t M = (size_t)s->M, o = (size_t)moff[p] * H;
        failed = failed || hsc[(size_t)p * 16 + 13] != 0.0;
        if (s->AHat) for (size_t m = 0; m < M; ++m) for (size_t h = 0; h < (size_t)H; ++h) s->AHat[h * M + m] = hA[o + m * H + h];
        if (s->SigmaA) memcpy(s->SigmaA, &hSA[p * HH], HH * 8);
        for (int64_t h = 0; h < H; ++h) {
            if (s->CA) s->CA[h + h * H] = hc[p * H + h];
            if (s->invCA) s->invCA[h + h * H] = hic[p * H + h];
        }
        if (s->YHat) memcpy(s->YHat, &hYH[(size_t)moff[p] * L], M * L * 8);
        s->sigma2 = hsc[(size_t)p * 16];
    }
    if (failed) { set_error("batched vbls: a posterior precision matrix was not positive definite (NaN written)"); return -2; }
    return 0;
}

// ---- K7 batched: lowerBound / lowerBoundTrimmed of many problems -------------------------------------------------------
static void lb_scalars(const vbmf_b200_sparse_state* s, Scalars& h) { h.alpha0p = s->alpha0; h.beta0p = s->beta0; h.alpha = s->alpha; }
static void lb_scalars(const vbmf_b200_dual_state* s, Scalars& h) {
    h.alpha00 = s->alpha00; h.beta00 = s->beta00; h.alpha01 = s->alpha01; h.beta01 = s->beta01;
    h.alpha_g0 = s->alpha0; h.alpha_g1 = s->alpha1;
}
static void lb_scalars(const vbmf_b200_trial_state* s, Scalars& h) {
    h.alpha00 = s->alpha01; h.beta00 = s->beta01; h.alpha01 = s->alpha02; h.beta01 = s->beta02; h.alpha02 = s->alpha03; h.beta02 = s->beta03;
    h.alpha_g0 = s->alpha1; h.alpha_g1 = s->alpha2; h.alpha_g2 = s->alpha3;
}

// Packs what the bound reads -- per column AHat, beta, CA, diag Sigma; per problem BHat, SigmaB, SigmaA, CB, delta and the
// scalars (the fields and the AHat / ATVecHat choice of the single solver's upload) -- into the batched path's staging arena.
template <class ST>
static int batched_lower_bound_impl(vbmf_b200_ctx* c, int kind, int64_t nprob, const double* const* Y, void* const* states,
                                    double trim, int trimmed, double* out) {
    if (nprob <= 0) return 0;
    const ST* s0 = (const ST*)states[0];
    if (s0 == nullptr) { set_error("batched lowerBound: NULL problem 0"); return -1; }
    const int64_t L = s0->L, H = s0->H;
    constexpr bool IS_DUAL = std::is_same<ST, vbmf_b200_dual_state>::value, IS_TRIAL = std::is_same<ST, vbmf_b200_trial_state>::value;
    int64_t H0 = H;
    if constexpr (IS_DUAL || IS_TRIAL) H0 = s0->H0;
    if (L < 1 || H < 1 || H > 64) { set_error("batched lowerBound supports 1 <= H <= 64 (got H = %lld)", (long long)H); return -1; }
    if (H0 < 0 || H0 > H) { set_error("H must be at least H0!"); return -1; }
    const int cw = vb::batched_lb_cols((int)H);
    std::vector<int> moff(nprob + 1, 0), coff(nprob + 1, 0), m0(nprob, 0);
    for (int64_t p = 0; p < nprob; ++p) {
        const ST* s = (const ST*)states[p];
        if (s == nullptr || Y[p] == nullptr) { set_error("batched lowerBound: NULL problem %lld", (long long)p); return -1; }
        if (s->L != L || s->H != H || s->M < 1 || s->M > 0x7fffff00LL) {
            set_error("batched lowerBound: problem %lld has different L/H or M < 1", (long long)p); return -1;
        }
        if constexpr (IS_DUAL || IS_TRIAL) { if (s->H0 != H0) { set_error("batched lowerBound: H0 differs"); return -1; } }
        if ((s->ATVecHat == nullptr && s->AHat == nullptr) || s->beta == nullptr || s->CA == nullptr || s->diagSigmaATVec == nullptr ||
            s->BHat == nullptr || s->SigmaB == nullptr || s->SigmaA == nullptr || s->CB == nullptr || s->delta == nullptr) {
            set_error("batched lowerBound: a required array of problem %lld is NULL", (long long)p); return -1;
        }
        if ((int64_t)moff[p] + s->M > 0x7fffff00LL) { set_error("batched lowerBound: more than 2^31 columns in one batch"); return -1; }
        moff[p + 1] = moff[p] + (int)s->M;
        coff[p + 1] = coff[p] + (int)((s->M + cw - 1) / cw);
        m0[p] = (int)s->M;
        if constexpr (IS_TRIAL) m0[p] = (int)std::min<int64_t>(std::max<int64_t>(s->M0, 0), s->M);
    }
    const int nch = coff[nprob];
    const size_t Mtot = (size_t)moff[nprob], MH = Mtot * H, HH = (size_t)H * H, LH = (size_t)L * H;
    VB_CUDA_OK(cudaSetDevice(c->device));
    // one arena: [inputs | result | device-only chunk partials]; one upload of the inputs, one download of the results
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += align_up(bytes, 256); return o; };
    const size_t o_moff = take((size_t)(nprob + 1) * 4), o_m0 = take((size_t)nprob * 4), o_coff = take((size_t)(nprob + 1) * 4),
                 o_cp = take((size_t)nch * 4), o_Y = take(L * Mtot * 8), o_A = take(MH * 8), o_beta = take(MH * 8), o_CA = take(MH * 8),
                 o_s = take(MH * 8), o_B = take(nprob * LH * 8), o_SB = take(nprob * HH * 8), o_SA = take(nprob * HH * 8),
                 o_CB = take(nprob * H * 8), o_dl = take(nprob * H * 8), o_sc = take((size_t)nprob * sizeof(Scalars));
    const size_t up_end = off;
    const size_t o_out = take((size_t)nprob * 8);
    const size_t o_part = take((size_t)nch * (vb::LB_NPART + HH) * 8);
    if (batch_reserve(c, off)) return -1;
    char* hb = c->batch_host;
    char* db = c->batch_dev;
    memcpy(hb + o_moff, moff.data(), (size_t)(nprob + 1) * 4);
    memcpy(hb + o_m0, m0.data(), (size_t)nprob * 4);
    memcpy(hb + o_coff, coff.data(), (size_t)(nprob + 1) * 4);
    int* hcp = (int*)(hb + o_cp);
    for (int64_t p = 0; p < nprob; ++p) for (int k = coff[p]; k < coff[p + 1]; ++k) hcp[k] = (int)p;
    double *hY = (double*)(hb + o_Y), *hA = (double*)(hb + o_A), *hbeta = (double*)(hb + o_beta), *hCA = (double*)(hb + o_CA),
           *hs = (double*)(hb + o_s), *hB = (double*)(hb + o_B), *hSB = (double*)(hb + o_SB), *hSA = (double*)(hb + o_SA),
           *hCB = (double*)(hb + o_CB), *hdl = (double*)(hb + o_dl);
    Scalars* hsc = (Scalars*)(hb + o_sc);
    parallel_for(nprob, [&](int64_t p) {
        const ST* s = (const ST*)states[p];
        const size_t M = (size_t)s->M, o = (size_t)moff[p] * H;
        memcpy(&hY[(size_t)moff[p] * L], Y[p], M * L * 8);
        if (s->ATVecHat) memcpy(&hA[o], s->ATVecHat, M * H * 8);      // up_A: ATVecHat when given, else AHat transposed
        else for (size_t m = 0; m < M; ++m) for (size_t h = 0; h < (size_t)H; ++h) hA[o + m * H + h] = s->AHat[h * M + m];
        memcpy(&hbeta[o], s->beta, M * H * 8);
        memcpy(&hCA[o], s->CA, M * H * 8);
        memcpy(&hs[o], s->diagSigmaATVec, M * H * 8);
        memcpy(&hB[p * LH], s->BHat, LH * 8);
        memcpy(&hSB[p * HH], s->SigmaB, HH * 8);
        memcpy(&hSA[p * HH], s->SigmaA, HH * 8);
        memcpy(&hCB[p * H], s->CB, H * 8);
        memcpy(&hdl[p * H], s->delta, H * 8);
        Scalars& h = hsc[p];                                          // sparse_like_upload + the kind's own upload
        memset(&h, 0, sizeof(Scalars));
        h.gamma0 = s->gamma0; h.delta0 = s->delta0; h.gamma = s->gamma;
        h.sigmaHat = s->sigmaHat; h.eta0 = s->eta0; h.zeta0 = s->zeta0; h.eta = s->eta; h.zeta = s->zeta;
        h.trYTY = s->trYTY;
        lb_scalars(s, h);
    });
    cudaStream_t st = c->st;
    if (cudaMemcpyAsync(db, hb, up_end, cudaMemcpyHostToDevice, st) != cudaSuccess) { cudaGetLastError(); set_error("batched lowerBound: upload failed"); return -1; }
    BatchLbDesc bd;
    bd.nprob = (int)nprob; bd.nchunk = nch; bd.L = (int)L; bd.H = (int)H; bd.H0 = (int)H0; bd.kind = kind; bd.trimmed = trimmed ? 1 : 0;
    bd.trim = trim;
    bd.moff = (const int*)(db + o_moff); bd.m0 = (const int*)(db + o_m0); bd.coff = (const int*)(db + o_coff); bd.cprob = (const int*)(db + o_cp);
    bd.Y = (const double*)(db + o_Y); bd.A = (const double*)(db + o_A); bd.beta = (const double*)(db + o_beta); bd.CA = (const double*)(db + o_CA);
    bd.sdiag = (const double*)(db + o_s); bd.B = (const double*)(db + o_B); bd.SigmaB = (const double*)(db + o_SB);
    bd.SigmaA = (const double*)(db + o_SA); bd.CB = (const double*)(db + o_CB); bd.delta = (const double*)(db + o_dl);
    bd.sc = (const Scalars*)(db + o_sc); bd.part = (double*)(db + o_part); bd.out = (double*)(db + o_out);
    prof_mark(c, c->ev_k1);       // profiling: the kernels alone (vbmf_b200_ctx_profile_read, K1 slot)
    int rc = k_batched_lower_bound(st, bd);
    prof_mark(c, c->ev_k1);
    if (!rc && cudaMemcpyAsync(hb + o_out, db + o_out, (size_t)nprob * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess) {
        cudaGetLastError(); set_error("batched lowerBound: download failed"); rc = -1;
    }
    { cudaError_t e = cudaStreamSynchronize(st); if (e != cudaSuccess && !rc) { set_error("batched lowerBound: %s", cudaGetErrorString(e)); rc = -1; } }
    if (rc) return rc;
    memcpy(out, hb + o_out, (size_t)nprob * 8);
    return 0;
}

extern "C" int vbmf_b200_batched_lower_bound(vbmf_b200_ctx* c, int kind, int64_t nprob, const double* const* Y, void* const* states,
                                             double trim, int trimmed, double* out) {
    if (!c || (nprob > 0 && (!Y || !states || !out))) { set_error("batched lowerBound: NULL argument"); return -1; }
    if (kind == VBMF_B200_SPARSE) return batched_lower_bound_impl<vbmf_b200_sparse_state>(c, kind, nprob, Y, states, trim, trimmed, out);
    if (kind == VBMF_B200_DUAL) return batched_lower_bound_impl<vbmf_b200_dual_state>(c, kind, nprob, Y, states, trim, trimmed, out);
    if (kind == VBMF_B200_TRIAL) return batched_lower_bound_impl<vbmf_b200_trial_state>(c, kind, nprob, Y, states, trim, trimmed, out);
    if (kind == VBMF_B200_DENSE) { set_error("the dense solver has no lowerBound (the reference defines none)"); return -1; }
    set_error("batched lowerBound: unknown parameter kind %d", kind);
    return -1;
}

extern "C" int vbmf_b200_batched_vbls(vbmf_b200_ctx* c, int kind, int64_t nprob, const double* const* Y, void* const* states,
                                      int64_t niter, int flags) {
    if (!c || (nprob > 0 && (!Y || !states))) { set_error("batched vbls: NULL argument"); return -1; }
    if (kind == VBMF_B200_SPARSE) return batched_vbls_impl<vbmf_b200_sparse_state>(c, kind, nprob, Y, states, niter, flags);
    if (kind == VBMF_B200_DUAL) return batched_vbls_impl<vbmf_b200_dual_state>(c, kind, nprob, Y, states, niter, flags);
    if (kind == VBMF_B200_TRIAL) return batched_vbls_impl<vbmf_b200_trial_state>(c, kind, nprob, Y, states, niter, flags);
    if (kind == VBMF_B200_DENSE) return batched_vbls_dense_impl(c, nprob, Y, states, niter);
    set_error("batched vbls: unknown parameter kind %d", kind);
    return -1;
}
