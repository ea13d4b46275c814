// gl_group: the multi-GPU plane of libgl_b200.so behind the C ABI (SURVEY 8b "an internal gl_group with an NCCL
// communicator", 8e).  #included at the end of gl_b200.cu (it uses that file's static helpers).
//
// One rank = one gl_ctx = one GPU.  A process may hold several ranks: a Rust prover drives every GPU of a box from one
// process (nlocal = nranks, no rendezvous token needed); torchrun-style launchers hold one rank per process and pass
// the token of gl_group_unique_id around out of band.  NCCL is bound at run time (dlopen "libnccl.so.2"): the library
// itself has no link-time dependency, a process that already loaded NCCL (torch) shares that copy, and every entry
// point other than gl_group_* works on a machine without NCCL.
//
// Sharding (SURVEY 8e): rank r owns leaf block r of nranks = LDE cosets k with bitrev_r(k) in that block = whole
// top-level Merkle subtrees + their cap entries (gl_ctx_set_shard).  Two exchanges carry data: the all-gather of
// coefficients (the IFFT is sharded by column: 1.13 GB in total at config 2, pipelined with the LDE; ncclAllGather for
// resident inputs, the ranks' own pull kernels over peer memory for host buffers: "coefficient exchange over peer memory"
// below) and the all-gather of the cap (512 B); the query openings of a proof are exchanged by gl_group_commit_open.
#include <dlfcn.h>
#include <nccl.h>
#include <sched.h>

#include <chrono>
#include <fstream>
#include <sstream>

namespace glnccl {
struct Api {
    void* so = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    ncclResult_t (*GetVersion)(int*) = nullptr;
    std::string error;
};
static Api* api() {
    static Api a;
    static std::once_flag once;
    std::call_once(once, [] {
        // 1. GL_B200_NCCL=<path> when set; 2. the copy this process already loaded (a host that imported torch shares
        // torch's bundled NCCL: two NCCLs with one SONAME in a process do not mix); 3. the system library.
        const char* forced = getenv("GL_B200_NCCL");
        if (forced && *forced) a.so = dlopen(forced, RTLD_NOW | RTLD_GLOBAL);
        if (!a.so) a.so = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
        for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
            if (a.so) break;
            a.so = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
        }
        if (!a.so) {
            a.error = std::string("NCCL is not available (dlopen libnccl.so.2): ") + (dlerror() ? dlerror() : "");
            return;
        }
        auto sym = [&](const char* n) {
            void* p = dlsym(a.so, n);
            if (!p && a.error.empty()) a.error = std::string("NCCL symbol missing: ") + n;
            return p;
        };
        a.GetUniqueId = (decltype(a.GetUniqueId))sym("ncclGetUniqueId");
        a.CommInitRank = (decltype(a.CommInitRank))sym("ncclCommInitRank");
        a.CommDestroy = (decltype(a.CommDestroy))sym("ncclCommDestroy");
        a.AllGather = (decltype(a.AllGather))sym("ncclAllGather");
        a.AllReduce = (decltype(a.AllReduce))sym("ncclAllReduce");
        a.GroupStart = (decltype(a.GroupStart))sym("ncclGroupStart");
        a.GroupEnd = (decltype(a.GroupEnd))sym("ncclGroupEnd");
        a.GetErrorString = (decltype(a.GetErrorString))sym("ncclGetErrorString");
        a.GetVersion = (decltype(a.GetVersion))sym("ncclGetVersion");
    });
    return &a;
}
}  // namespace glnccl

struct gl_group_rank {
    gl_ctx* ctx = nullptr;
    ncclComm_t comm = nullptr;
    cudaStream_t comm_stream = nullptr;
    cudaStream_t prep_stream = nullptr;   // uploads' consumers: the rank's own copy-in + IFFT of every round, ahead of the LDE queue
    std::vector<cudaEvent_t> ev;   // per round: [2j] own coefficients ready, [2j+1] round gathered; + tail events
    u64* cap_all = nullptr;        // [2^cap_height][4] gathered cap (device)
    size_t cap_all_bytes = 0;
    u64* open_buf = nullptr;       // [k][c + 4 L] rows + paths exchanged by gl_group_commit_open
    size_t open_bytes = 0;
    // peer-memory plane (see "coefficient exchange over peer memory" below)
    u64* xbuf = nullptr;           // this rank's exchange buffer: [XB_FLAGS] ready flags, then its published coefficient slices
    std::vector<u64*> peer_x;      // [nranks]: every rank's xbuf as this device addresses it (own rank: xbuf)
    std::vector<char> peer_ipc;    // 1 = opened with cudaIpcOpenMemHandle
    u64** d_peer_x = nullptr;      // the same table on the device
};
struct gl_group {
    uint32_t nlocal = 0, rank0 = 0, nranks = 1;
    std::vector<gl_group_rank> r;
    std::string err;
    std::mutex mu;
    float phase_ms[GL_PHASES] = {};
    // coefficient exchange over peer memory: -1 = not tried yet, 0 = NCCL all-gather, 1 = pull kernels over NVLink
    int p2p = -1;
    size_t xbuf_words = 0;         // capacity of every rank's exchange buffer (the same everywhere)
    uint64_t epoch = 0;            // commits made with the peer-memory exchange; the value the ready flags carry
};

static void group_unmap_peers(gl_group* g);

static int gfail(gl_group* g, int code, const std::string& msg) {
    if (g) g->err = msg;
    else g_create_error = msg;
    return code;
}
#define NCK(g, call)                                                                                         \
    do {                                                                                                     \
        ncclResult_t r__ = (call);                                                                           \
        if (r__ != ncclSuccess)                                                                              \
            return gfail(g, GL_E_NCCL, std::string(#call) + ": " + glnccl::api()->GetErrorString(r__));      \
    } while (0)
#define GCK(g, call)                                                                                         \
    do {                                                                                                     \
        cudaError_t e__ = (call);                                                                            \
        if (e__ != cudaSuccess) {                                                                            \
            cudaGetLastError();                                                                              \
            return gfail(g, GL_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));                 \
        }                                                                                                    \
    } while (0)
// a single-ctx helper failed: carry its message to the group
#define GTRY(g, ctx, expr)                              \
    do {                                                \
        int rc__ = (expr);                              \
        if (rc__) return gfail(g, rc__, (ctx)->err);    \
    } while (0)

extern "C" int gl_group_unique_id(uint8_t* id_out) {
    if (!id_out) return gfail(nullptr, GL_E_ARG, "gl_group_unique_id: NULL");
    auto* a = glnccl::api();
    if (!a->error.empty()) return gfail(nullptr, GL_E_NCCL, a->error);
    static_assert(sizeof(ncclUniqueId) == GL_GROUP_ID_BYTES, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    ncclResult_t r = a->GetUniqueId(&id);
    if (r != ncclSuccess) return gfail(nullptr, GL_E_NCCL, std::string("ncclGetUniqueId: ") + a->GetErrorString(r));
    memcpy(id_out, &id, sizeof id);
    return GL_OK;
}

extern "C" void gl_group_destroy(gl_group* g) {
    if (!g) return;
    auto* a = glnccl::api();
    for (auto& rk : g->r) {
        if (!rk.ctx) continue;
        cudaSetDevice(rk.ctx->device);
        cudaStreamSynchronize(rk.ctx->stream);
        if (rk.comm_stream) cudaStreamSynchronize(rk.comm_stream);
    }
    group_unmap_peers(g);
    for (auto& rk : g->r) {
        if (!rk.ctx) continue;
        Guard gd(rk.ctx);
        cudaSetDevice(rk.ctx->device);
        if (rk.xbuf) cudaFree(rk.xbuf);
        if (rk.d_peer_x) cudaFree(rk.d_peer_x);
        cudaStreamSynchronize(rk.ctx->stream);
        if (rk.comm_stream) cudaStreamSynchronize(rk.comm_stream);
        if (rk.comm && a->CommDestroy) a->CommDestroy(rk.comm);
        for (auto e : rk.ev) cudaEventDestroy(e);
        if (rk.cap_all) cudaFree(rk.cap_all);
        if (rk.open_buf) cudaFree(rk.open_buf);
        if (rk.comm_stream) cudaStreamDestroy(rk.comm_stream);
        if (rk.prep_stream) cudaStreamDestroy(rk.prep_stream);
        rk.ctx->shard_index = 0;
        rk.ctx->shard_count = 1;
    }
    delete g;
}

extern "C" int gl_group_create(gl_ctx* const* ctxs, uint32_t nlocal, uint32_t rank0, uint32_t nranks, const uint8_t* id,
                               gl_group** out) {
    if (!out) return gfail(nullptr, GL_E_ARG, "gl_group_create: out is NULL");
    *out = nullptr;
    if (!ctxs || nlocal == 0 || !is_pow2(nranks) || rank0 + (uint64_t)nlocal > nranks)
        return gfail(nullptr, GL_E_ARG, "gl_group_create: nranks must be a power of two and rank0 + nlocal <= nranks");
    if (!id && nlocal != nranks)
        return gfail(nullptr, GL_E_ARG, "gl_group_create: a group that spans processes needs the token of gl_group_unique_id");
    for (uint32_t i = 0; i < nlocal; i++) {
        if (!ctxs[i]) return gfail(nullptr, GL_E_ARG, "gl_group_create: NULL context");
        for (uint32_t j = 0; j < i; j++)
            if (ctxs[j]->device == ctxs[i]->device) return gfail(nullptr, GL_E_ARG, "gl_group_create: one rank per GPU (two contexts share a device)");
    }
    auto* a = glnccl::api();
    if (!a->error.empty()) return gfail(nullptr, GL_E_NCCL, a->error);
    gl_group* g = new (std::nothrow) gl_group();
    if (!g) return gfail(nullptr, GL_E_OOM, "host allocation failed");
    g->nlocal = nlocal; g->rank0 = rank0; g->nranks = nranks;
    g->r.resize(nlocal);
    ncclUniqueId uid;
    if (id) memcpy(&uid, id, sizeof uid);
    else {
        ncclResult_t r = a->GetUniqueId(&uid);
        if (r != ncclSuccess) { delete g; return gfail(nullptr, GL_E_NCCL, std::string("ncclGetUniqueId: ") + a->GetErrorString(r)); }
    }
    int prev = -1;
    cudaGetDevice(&prev);
    int rc = GL_OK;
    std::string msg;
    if (nranks > 1) {
        // all local ranks join in one NCCL group call (required when one thread initialises several devices)
        ncclResult_t r = a->GroupStart();
        for (uint32_t i = 0; i < nlocal && r == ncclSuccess; i++) {
            cudaSetDevice(ctxs[i]->device);
            r = a->CommInitRank(&g->r[i].comm, (int)nranks, uid, (int)(rank0 + i));
        }
        ncclResult_t r2 = a->GroupEnd();
        if (r == ncclSuccess) r = r2;
        if (r != ncclSuccess) { rc = GL_E_NCCL; msg = std::string("ncclCommInitRank: ") + a->GetErrorString(r); }
    }
    for (uint32_t i = 0; i < nlocal && rc == GL_OK; i++) {
        cudaSetDevice(ctxs[i]->device);
        // highest priority: the block scheduler places the collective's few CTAs ahead of the thousands of queued LDE /
        // hashing CTAs of the compute stream, so a gather is on the wire as soon as its data exists instead of when the
        // running compute kernel drains (measured at 8 GPUs: gather 0 finished at 3.0 ms instead of 0.8 ms without this)
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        cudaError_t e = cudaStreamCreateWithPriority(&g->r[i].comm_stream, cudaStreamNonBlocking, hi);
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&g->r[i].prep_stream, cudaStreamNonBlocking, hi);
        if (e != cudaSuccess) { rc = GL_E_CUDA; msg = std::string("cudaStreamCreate: ") + cudaGetErrorString(e); }
    }
    if (prev >= 0) cudaSetDevice(prev);
    if (rc != GL_OK) {
        for (auto& rk : g->r) {
            if (rk.comm) a->CommDestroy(rk.comm);
            if (rk.comm_stream) cudaStreamDestroy(rk.comm_stream);
            if (rk.prep_stream) cudaStreamDestroy(rk.prep_stream);
        }
        delete g;
        return gfail(nullptr, rc, msg);
    }
    for (uint32_t i = 0; i < nlocal; i++) {
        g->r[i].ctx = ctxs[i];
        ctxs[i]->shard_index = rank0 + i;
        ctxs[i]->shard_count = nranks;
    }
    *out = g;
    return GL_OK;
}

extern "C" const char* gl_group_last_error(const gl_group* g) { return g ? g->err.c_str() : g_create_error.c_str(); }
extern "C" int gl_group_info(const gl_group* g, uint32_t* nlocal, uint32_t* rank0, uint32_t* nranks, int* nccl_version) {
    if (!g) return GL_E_ARG;
    if (nlocal) *nlocal = g->nlocal;
    if (rank0) *rank0 = g->rank0;
    if (nranks) *nranks = g->nranks;
    if (nccl_version) {
        *nccl_version = 0;
        if (glnccl::api()->GetVersion) glnccl::api()->GetVersion(nccl_version);
    }
    return GL_OK;
}
extern "C" int gl_group_commit_phase_ms(const gl_group* g, float* out6) {
    if (!g || !out6) return GL_E_ARG;
    for (int i = 0; i < GL_PHASES; i++) out6[i] = g->phase_ms[i];
    return GL_OK;
}

// Host threads of the calling process next to the GPU: pins the CALLING thread (and the memory it first-touches or
// page-locks afterwards) to the CPUs of the NUMA node the device hangs off (sysfs local_cpulist of its PCI function).
extern "C" int gl_ctx_bind_host_numa(gl_ctx* ctx) {
    if (!ctx) return GL_E_ARG;
    char bus[32] = {};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, ctx->device) != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, GL_E_CUDA, "gl_ctx_bind_host_numa: no PCI bus id");
    }
    for (char* p = bus; *p; p++) *p = (char)tolower(*p);
    std::ifstream f(std::string("/sys/bus/pci/devices/") + bus + "/local_cpulist");
    std::string list;
    if (!f || !std::getline(f, list) || list.empty()) return fail(ctx, GL_E_STATE, "gl_ctx_bind_host_numa: no local_cpulist for " + std::string(bus));
    cpu_set_t set;
    CPU_ZERO(&set);
    std::stringstream ss(list);
    std::string tok;
    int count = 0;
    while (std::getline(ss, tok, ',')) {
        int lo = 0, hi = 0;
        if (sscanf(tok.c_str(), "%d-%d", &lo, &hi) == 2) {
        } else if (sscanf(tok.c_str(), "%d", &lo) == 1) hi = lo;
        else continue;
        for (int c = lo; c <= hi && c < CPU_SETSIZE; c++) { CPU_SET(c, &set); count++; }
    }
    if (!count) return fail(ctx, GL_E_STATE, "gl_ctx_bind_host_numa: empty local_cpulist");
    cpu_set_t allowed;
    if (sched_getaffinity(0, sizeof allowed, &allowed) == 0) {
        cpu_set_t both;
        CPU_AND(&both, &set, &allowed);
        if (CPU_COUNT(&both) == 0) return fail(ctx, GL_E_STATE, "gl_ctx_bind_host_numa: the device's CPUs are outside this process's affinity mask");
        set = both;
    }
    if (sched_setaffinity(0, sizeof set, &set) != 0) return fail(ctx, GL_E_STATE, "gl_ctx_bind_host_numa: sched_setaffinity failed");
    return GL_OK;
}

// ---- coefficient exchange over peer memory -------------------------------------------------------------------------------
// The all-gather of the inverse-transformed polynomials as the ranks' OWN kernels over NVLink / NVSwitch peer memory
// instead of ncclAllGather.  Every rank owns an exchange buffer that every other rank maps (cudaIpcOpenMemHandle across
// processes, cudaDeviceEnablePeerAccess inside one).  Round j: the owner copies its slice into the buffer and raises
// ready flag j to the commit's epoch (k_group_signal: system-scope fence, then the store); its peers' pull kernels wait on
// that flag THROUGH the mapping and then stream the slice into their own coefficient array with 16-byte loads that bypass
// L1 (the line's home is the owner's L2).  No host thread and no copy engine takes part, so the exchange neither waits
// for nor slows the host<->device DMA of the end-to-end path, and a rank starts pulling from each peer the moment that
// peer has published, not when the slowest one has.  Reuse of the buffer across commits is safe because every commit ends
// with the cap all-gather: a rank passes it only after every rank has built its tree, i.e. finished all its pulls.
#define XB_FLAGS 64u   // u64 words reserved for ready flags (rounds per commit <= 64)

__global__ void k_group_signal(u64* flag, u64 value) {
    __threadfence_system();
    *reinterpret_cast<volatile u64*>(flag) = value;
}
// grid (CTAs per peer, nranks): blockIdx.y = the rank pulled from.  src_words: offset of the round's slice in a peer's
// exchange buffer; dst: this rank's [nranks][count] block of the round (slot p receives rank p's slice).
__global__ void __launch_bounds__(256)
k_group_pull(u64* const* __restrict__ peer_x, u32 me, u32 flag_index, u64 epoch, u64 src_words, u64* __restrict__ dst, u64 count) {
    const u32 p = blockIdx.y;
    if (p == me) return;
    const u64* px = peer_x[p];
    if (threadIdx.x == 0) {
        const volatile u64* f = px + flag_index;
        while (*f < epoch) __nanosleep(100);
        __threadfence_system();
    }
    __syncthreads();
    const uint4* src = reinterpret_cast<const uint4*>(px + src_words);
    uint4* out = reinterpret_cast<uint4*>(dst + (u64)p * count);
    const u64 vecs = count >> 1, stride = (u64)gridDim.x * 256;
    u64 i = blockIdx.x * (u64)256 + threadIdx.x;
    for (; i + 3 * stride < vecs; i += 4 * stride) {
        const uint4 a = __ldcg(src + i), b = __ldcg(src + i + stride), c = __ldcg(src + i + 2 * stride), d = __ldcg(src + i + 3 * stride);
        out[i] = a; out[i + stride] = b; out[i + 2 * stride] = c; out[i + 3 * stride] = d;
    }
    for (; i < vecs; i += stride) out[i] = __ldcg(src + i);
}

static void group_unmap_peers(gl_group* g) {
    for (auto& rk : g->r) {
        if (!rk.ctx) continue;
        cudaSetDevice(rk.ctx->device);
        for (size_t r = 0; r < rk.peer_x.size(); r++)
            if (rk.peer_ipc[r] && rk.peer_x[r]) cudaIpcCloseMemHandle(rk.peer_x[r]);
        rk.peer_x.clear();
        rk.peer_ipc.clear();
    }
}
// Collective.  Makes sure every rank has an exchange buffer of at least `words` and a mapping of everybody else's; decides
// ONCE, for the whole group, whether the peer-memory exchange is used (g->p2p).
static int group_ensure_exchange(gl_group* g, size_t words) {
    auto* a = glnccl::api();
    const uint32_t G = g->nranks, nl = g->nlocal;
    if (g->p2p == 0) return GL_OK;
    if (g->p2p == 1 && g->xbuf_words >= words) return GL_OK;
    // every rank reaches this point for the same commit (same geometry => same `words`): (re)build the plane together
    for (auto& rk : g->r) {
        cudaSetDevice(rk.ctx->device);
        cudaStreamSynchronize(rk.ctx->stream);
        cudaStreamSynchronize(rk.comm_stream);
    }
    group_unmap_peers(g);
    const size_t cap = words + words / 4;
    int ok = 1;
    std::vector<cudaIpcMemHandle_t> mine(nl);
    for (uint32_t i = 0; i < nl; i++) {
        gl_group_rank& rk = g->r[i];
        cudaSetDevice(rk.ctx->device);
        if (rk.xbuf) cudaFree(rk.xbuf);
        rk.xbuf = nullptr;
        if (cudaMalloc(&rk.xbuf, cap * 8) != cudaSuccess || cudaMemset(rk.xbuf, 0, XB_FLAGS * 8) != cudaSuccess ||
            cudaIpcGetMemHandle(&mine[i], rk.xbuf) != cudaSuccess) {
            cudaGetLastError();
            ok = 0;
        }
        if (!rk.d_peer_x && cudaMalloc(&rk.d_peer_x, G * sizeof(u64*)) != cudaSuccess) { cudaGetLastError(); ok = 0; }
    }
    // handles of all ranks (NCCL as the bootstrap: one small all-gather per local rank)
    const size_t hb = sizeof(cudaIpcMemHandle_t);
    std::vector<unsigned char*> d_h(nl, nullptr);
    std::vector<std::vector<unsigned char>> all(nl, std::vector<unsigned char>(G * hb));
    for (uint32_t i = 0; i < nl; i++) {
        cudaSetDevice(g->r[i].ctx->device);
        if (cudaMalloc(&d_h[i], G * hb) != cudaSuccess) { cudaGetLastError(); return gfail(g, GL_E_OOM, "gl_group: exchange set-up allocation failed"); }
        cudaMemcpy(d_h[i] + (size_t)(g->rank0 + i) * hb, &mine[i], hb, cudaMemcpyHostToDevice);
    }
    if (nl > 1) NCK(g, a->GroupStart());
    for (uint32_t i = 0; i < nl; i++) {
        cudaSetDevice(g->r[i].ctx->device);
        ncclResult_t r = a->AllGather(d_h[i] + (size_t)(g->rank0 + i) * hb, d_h[i], hb, ncclUint8, g->r[i].comm, g->r[i].comm_stream);
        if (r != ncclSuccess) {
            if (nl > 1) a->GroupEnd();
            return gfail(g, GL_E_NCCL, std::string("ncclAllGather (exchange handles): ") + a->GetErrorString(r));
        }
    }
    if (nl > 1) NCK(g, a->GroupEnd());
    for (uint32_t i = 0; i < nl; i++) {
        cudaSetDevice(g->r[i].ctx->device);
        cudaStreamSynchronize(g->r[i].comm_stream);
        cudaMemcpy(all[i].data(), d_h[i], G * hb, cudaMemcpyDeviceToHost);
        cudaFree(d_h[i]);
    }
    for (uint32_t i = 0; i < nl && ok; i++) {
        gl_group_rank& rk = g->r[i];
        cudaSetDevice(rk.ctx->device);
        rk.peer_x.assign(G, nullptr);
        rk.peer_ipc.assign(G, 0);
        for (uint32_t r = 0; r < G && ok; r++) {
            if (r >= g->rank0 && r < g->rank0 + nl) {           // a rank of this process: its pointer, with peer access
                gl_group_rank& other = g->r[r - g->rank0];
                if (r != g->rank0 + i) {
                    int can = 0;
                    cudaDeviceCanAccessPeer(&can, rk.ctx->device, other.ctx->device);
                    cudaError_t pe = can ? cudaDeviceEnablePeerAccess(other.ctx->device, 0) : cudaErrorInvalidDevice;
                    if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) ok = 0;
                    cudaGetLastError();
                }
                rk.peer_x[r] = other.xbuf;
            } else {
                cudaIpcMemHandle_t h;
                memcpy(&h, all[i].data() + (size_t)r * hb, hb);
                void* ptr = nullptr;
                if (cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                    cudaGetLastError();
                    ok = 0;
                } else {
                    rk.peer_x[r] = (u64*)ptr;
                    rk.peer_ipc[r] = 1;
                }
            }
        }
        if (ok && cudaMemcpy(rk.d_peer_x, rk.peer_x.data(), G * sizeof(u64*), cudaMemcpyHostToDevice) != cudaSuccess) { cudaGetLastError(); ok = 0; }
    }
    // one decision for the whole group: the minimum of the ranks' outcomes
    std::vector<u64*> d_ok(nl, nullptr);
    for (uint32_t i = 0; i < nl; i++) {
        cudaSetDevice(g->r[i].ctx->device);
        const u64 v = (u64)ok;
        if (cudaMalloc(&d_ok[i], 8) != cudaSuccess) { cudaGetLastError(); return gfail(g, GL_E_OOM, "gl_group: exchange set-up allocation failed"); }
        cudaMemcpy(d_ok[i], &v, 8, cudaMemcpyHostToDevice);
    }
    if (nl > 1) NCK(g, a->GroupStart());
    for (uint32_t i = 0; i < nl; i++) {
        cudaSetDevice(g->r[i].ctx->device);
        ncclResult_t r = a->AllReduce(d_ok[i], d_ok[i], 1, ncclUint64, ncclMin, g->r[i].comm, g->r[i].comm_stream);
        if (r != ncclSuccess) {
            if (nl > 1) a->GroupEnd();
            return gfail(g, GL_E_NCCL, std::string("ncclAllReduce (exchange set-up): ") + a->GetErrorString(r));
        }
    }
    if (nl > 1) NCK(g, a->GroupEnd());
    u64 all_ok = 1;
    for (uint32_t i = 0; i < nl; i++) {
        cudaSetDevice(g->r[i].ctx->device);
        cudaStreamSynchronize(g->r[i].comm_stream);
        u64 v = 0;
        cudaMemcpy(&v, d_ok[i], 8, cudaMemcpyDeviceToHost);
        cudaFree(d_ok[i]);
        if (!v) all_ok = 0;
    }
    if (!all_ok) {   // no peer access somewhere: everybody stays on ncclAllGather
        group_unmap_peers(g);
        for (auto& rk : g->r) {
            cudaSetDevice(rk.ctx->device);
            if (rk.xbuf) cudaFree(rk.xbuf);
            rk.xbuf = nullptr;
        }
        g->p2p = 0;
        g->xbuf_words = 0;
        return GL_OK;
    }
    g->p2p = 1;
    g->xbuf_words = cap;
    return GL_OK;
}

// ---- the collective commit ---------------------------------------------------------------------------------------
// Column plan: round 0 holds ONE polynomial per rank (nothing can run under its IFFT + gather, so it is short), the
// others W each; round j occupies the padded columns [base_j, base_j + nranks * w_j) and rank r inverse-transforms the
// slice [base_j + r * w_j, + w_j): an in-place ncclAllGather per round completes the block on every rank.
struct GroupPlan {
    uint32_t rounds = 0, cpad = 0;
    std::vector<uint32_t> base, w;
};
static GroupPlan group_plan(uint32_t c, uint32_t nranks) {
    GroupPlan p;
    const uint32_t target_rounds = 5;
    uint32_t rest = c > nranks ? c - nranks : 0;
    uint32_t W = (rest + nranks * (target_rounds - 1) - 1) / (nranks * (target_rounds - 1));
    if (W < 1) W = 1;
    uint32_t at = 0;
    while (at < c) {
        uint32_t wj = p.rounds == 0 ? 1 : W;
        p.base.push_back(at);
        p.w.push_back(wj);
        at += wj * nranks;
        p.rounds++;
    }
    p.cpad = at;
    return p;
}
static inline uint32_t clampc(uint32_t x, uint32_t c) { return x < c ? x : c; }

// GL_B200_TRACE=1: device-side timeline of one collective commit (ms after its first event), rank by rank, on stderr
struct GroupTrace {
    bool on = false;
    std::vector<std::pair<std::string, cudaEvent_t>> marks;
    std::vector<std::pair<std::string, double>> host;   // when the host thread ENQUEUED the step (ms after the first mark)
    std::chrono::steady_clock::time_point t0;
    void mark(const std::string& name, cudaStream_t st) {
        if (!on) return;
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) return;
        cudaEventRecord(e, st);
        if (marks.empty() && host.empty()) t0 = std::chrono::steady_clock::now();
        host.emplace_back(name, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
        marks.emplace_back(name, e);
    }
    void dump(uint32_t rank, cudaEvent_t origin) {
        if (!on) return;
        std::string line = "[gl_group trace] rank " + std::to_string(rank) + ":";
        for (auto& m : marks) {
            float ms = 0;
            cudaEventElapsedTime(&ms, origin, m.second);
            char buf[64];
            snprintf(buf, sizeof buf, " %s=%.2f", m.first.c_str(), ms);
            line += buf;
            cudaEventDestroy(m.second);
        }
        line += " | enqueued:";
        for (auto& h : host) {
            char buf[64];
            snprintf(buf, sizeof buf, " %s=%.2f", h.first.c_str(), h.second);
            line += buf;
        }
        fprintf(stderr, "%s\n", line.c_str());
        marks.clear();
        host.clear();
    }
};

static int group_commit(gl_group* g, const uint64_t* const* inputs, bool is_values, uint32_t log_n, uint32_t c,
                        uint32_t rate_bits, uint32_t cap_height, uint64_t* const* coeffs_out, uint64_t* const* cap_out,
                        gl_commit** handles, int space, uint32_t flags, const char* name) {
    if (!g) return GL_E_ARG;
    if (!inputs || !handles) return gfail(g, GL_E_ARG, std::string(name) + ": NULL argument");
    std::lock_guard<std::mutex> lk(g->mu);
    std::vector<std::unique_lock<std::mutex>> ctx_locks;   // calls on one ctx are serialised (as Guard does)
    for (auto& rk : g->r) ctx_locks.emplace_back(rk.ctx->mu);
    auto* a = glnccl::api();
    const uint32_t G = g->nranks, nl = g->nlocal;
    for (uint32_t i = 0; i < nl; i++) {
        handles[i] = nullptr;
        if (!inputs[i]) return gfail(g, GL_E_ARG, std::string(name) + ": NULL polynomials");
        gl_ctx* ctx = g->r[i].ctx;
        GTRY(g, ctx, commit_check(ctx, log_n, c, rate_bits, cap_height, name));
        const std::string nm(name), rank = "[" + std::to_string(i) + "]";
        const size_t bytes = ((size_t)c << log_n) * 8;
        GTRY(g, ctx, check_device_ptr(ctx, space, inputs[i], bytes, (nm + (is_values ? ": values" : ": coeffs") + rank).c_str()));
        if (coeffs_out) GTRY(g, ctx, check_device_ptr(ctx, space, coeffs_out[i], bytes, (nm + ": coeffs_out" + rank).c_str()));
        if (cap_out) GTRY(g, ctx, check_device_ptr(ctx, space, cap_out[i], (size_t)32 << cap_height, (nm + ": cap_out" + rank).c_str()));
    }
    const u64 n = (u64)1 << log_n;
    const GroupPlan plan = group_plan(c, G);
    const size_t cap_bytes = (size_t)32 << cap_height;
    // this rank's slices of all rounds, published one after the other behind the flags of its exchange buffer
    std::vector<u64> xoff(plan.rounds + 1, XB_FLAGS);
    for (uint32_t j = 0; j < plan.rounds; j++) xoff[j + 1] = xoff[j] + (u64)plan.w[j] * n;
    // Which exchange: with host buffers the rounds arrive at the pace of PCIe and the pull kernels, which take each peer's
    // slice the moment it is published and share nothing with the DMA engines, win (8 GPUs: 22.4 against 24.1 ms end to
    // end); with everything resident ncclAllGather's few CTAs disturb the hashing slightly less (15.7 against 15.9 ms).
    // GL_B200_GROUP_P2P = 0: NCCL always, 2: pull kernels always.
    static const int p2p_mode = getenv("GL_B200_GROUP_P2P") ? atoi(getenv("GL_B200_GROUP_P2P")) : 1;
    const bool want_p2p = G > 1 && plan.rounds <= XB_FLAGS && log_n >= 1 &&   // 16-byte copies: two coefficients at least
                          (p2p_mode == 2 || (p2p_mode == 1 && space == GL_HOST));
    if (want_p2p) {
        int rc = group_ensure_exchange(g, (size_t)xoff[plan.rounds]);
        if (rc != GL_OK) return rc;
    }
    const bool p2p = want_p2p && g->p2p == 1;
    if (p2p) g->epoch++;
    std::vector<GroupTrace> trace(nl);
    {
        const char* t = getenv("GL_B200_TRACE");
        for (auto& tr : trace) tr.on = t && t[0] == '1';
    }
    int prev = -1;
    cudaGetDevice(&prev);
    struct Restore { int d; ~Restore() { if (d >= 0) cudaSetDevice(d); } } restore{prev};
    // Handles still held when this function returns belong to a failed commit.  `bail` drops them rank by rank, with the
    // rank's device current, once nothing the rank queued (its streams, the coefficient downloads) can use their blocks.
    std::vector<std::unique_ptr<gl_commit>> hs(nl);
    struct Bail {
        gl_group* g;
        std::vector<std::unique_ptr<gl_commit>>& hs;
        int space;
        ~Bail() {
            for (uint32_t i = 0; i < hs.size(); i++) {
                if (!hs[i]) continue;
                gl_ctx* ctx = g->r[i].ctx;
                cudaSetDevice(ctx->device);
                if (space == GL_HOST) downloads_wait(ctx);
                cudaStreamSynchronize(g->r[i].comm_stream);
                cudaStreamSynchronize(g->r[i].prep_stream);
                quiesce(ctx);
                hs[i].reset();
            }
        }
    } bail{g, hs, space};
    // ---- allocate
    for (uint32_t i = 0; i < nl; i++) {
        gl_group_rank& rk = g->r[i];
        gl_ctx* ctx = rk.ctx;
        GCK(g, cudaSetDevice(ctx->device));
        // every rank salts its own leaves
        GTRY(g, ctx, commit_new(ctx, log_n, c, rate_bits, cap_height, (flags & GL_COMMIT_BLINDING) ? GL_SALT_SIZE : 0, plan.cpad,
                                &hs[i]));
        gl_commit* h = hs[i].get();
        h->stream_hash = (flags & GL_COMMIT_STREAM_HASH) && c > 4 && !h->salt;
        while (rk.ev.size() < 2 * (size_t)plan.rounds + 2) {
            cudaEvent_t e;
            cudaError_t ce = cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
            if (ce != cudaSuccess) return gfail(g, GL_E_CUDA, cudaGetErrorString(ce));
            rk.ev.push_back(e);
        }
        if (rk.cap_all_bytes < cap_bytes) {
            if (rk.cap_all) cudaFree(rk.cap_all);
            rk.cap_all = nullptr;
            cudaError_t ce = cudaMalloc(&rk.cap_all, cap_bytes);
            if (ce != cudaSuccess) return gfail(g, GL_E_OOM, cudaGetErrorString(ce));
            rk.cap_all_bytes = cap_bytes;
        }
        // the padding columns of the last round take part in the gather: keep them defined
        if (plan.cpad > c) {
            // only the ranks' own padded slices are sent; zero them
            const uint32_t j = plan.rounds - 1;
            const uint32_t own0 = plan.base[j] + (g->rank0 + i) * plan.w[j], own1 = own0 + plan.w[j];
            const uint32_t z0 = own0 > c ? own0 : c;
            if (own1 > z0) cudaMemsetAsync(h->coeffs.get() + (size_t)z0 * n, 0, (size_t)(own1 - z0) * n * 8, ctx->stream);
        }
        for (int e = 0; e <= 3; e++) mark(ctx, e);
    }
    // ---- rounds: IFFT(j) is issued before LDE(j - 1) so that gather j is on the wire while round j - 1 is extended
    auto lde_round = [&](uint32_t i, uint32_t j) -> int {
        gl_group_rank& rk = g->r[i];
        gl_ctx* ctx = rk.ctx;
        gl_commit* h = hs[i].get();
        cudaSetDevice(ctx->device);
        cudaError_t ce = cudaStreamWaitEvent(ctx->stream, rk.ev[2 * j + 1], 0);
        if (ce != cudaSuccess) return gfail(g, GL_E_CUDA, cudaGetErrorString(ce));
        const uint32_t c0 = plan.base[j], c1 = clampc(c0 + plan.w[j] * G, c);
        if (c1 > c0) {
            int rc = commit_lde_columns(ctx, h, c0, c1 - c0);
            trace[i].mark("lde" + std::to_string(j), ctx->stream);
            if (rc == GL_OK) rc = commit_absorb_block(ctx, h, c0, c1 - c0);
            if (h->stream_hash) trace[i].mark("abs" + std::to_string(j), ctx->stream);
            if (rc != GL_OK) return gfail(g, rc, ctx->err);
        }
        return GL_OK;
    };
    std::vector<staging::HostSeg> segs;
    for (uint32_t j = 0; j < plan.rounds; j++) {
        for (uint32_t i = 0; i < nl; i++) {
            gl_group_rank& rk = g->r[i];
            gl_ctx* ctx = rk.ctx;
            gl_commit* h = hs[i].get();
            GCK(g, cudaSetDevice(ctx->device));
            const uint32_t own0 = plan.base[j] + (g->rank0 + i) * plan.w[j];
            const uint32_t o0 = clampc(own0, c), o1 = clampc(own0 + plan.w[j], c);
            // This rank's copy-in + IFFT of round j run on the prep stream: they start when the upload lands, not when
            // the LDE / hashing of earlier rounds queued on the main stream has drained, so the exchange of round j is
            // never held up by the compute backlog (and the main stream never waits for an upload it does not need yet).
            struct StreamSwap {
                gl_ctx* c; cudaStream_t saved;
                StreamSwap(gl_ctx* c_, cudaStream_t s) : c(c_), saved(c_->stream) { c->stream = s; }
                ~StreamSwap() { c->stream = saved; }
            } on_prep(ctx, rk.prep_stream);
            if (j == 0) cudaStreamWaitEvent(rk.prep_stream, ctx->ev[3], 0);   // buffers allocated / padded on the main stream
            if (o1 > o0) {
                u64* dcol = h->coeffs.get() + (size_t)o0 * n;
                const size_t bytes = (size_t)(o1 - o0) * n * 8;
                if (space == GL_DEVICE) {
                    cudaError_t ce = cudaMemcpyAsync(dcol, inputs[i] + (size_t)o0 * n, bytes, cudaMemcpyDeviceToDevice, ctx->stream);
                    if (ce != cudaSuccess) return gfail(g, GL_E_CUDA, cudaGetErrorString(ce));
                } else {
                    if (j == 0) cudaStreamWaitEvent(ctx->h2d_stream, ctx->ev[0], 0);
                    GTRY(g, ctx, h2d_copy(ctx, dcol, inputs[i] + (size_t)o0 * n, bytes, ctx->h2d_stream));
                    cudaEventRecord(rk.ev[2 * j], ctx->h2d_stream);
                    cudaStreamWaitEvent(ctx->stream, rk.ev[2 * j], 0);
                    trace[i].mark("up" + std::to_string(j), ctx->h2d_stream);
                }
                if (is_values)   // "IFFT" of this rank's columns
                    GTRY(g, ctx, transform_natural(ctx, dcol, log_n, o1 - o0, true, nullptr, nullptr));
            }
            cudaEventRecord(rk.ev[2 * j], ctx->stream);
            trace[i].mark("ifft" + std::to_string(j), ctx->stream);
            if (o1 > o0 && is_values && coeffs_out && coeffs_out[i] && space == GL_HOST)
                GTRY(g, ctx, d2h_copy(ctx, {staging::HostSeg{coeffs_out[i] + (size_t)o0 * n, (size_t)(o1 - o0) * n * 8}},
                                      h->coeffs.get() + (size_t)o0 * n, rk.ev[2 * j]));
            cudaStreamWaitEvent(rk.comm_stream, rk.ev[2 * j], 0);
        }
        if (p2p) {
            // publish: own slice into the exchange buffer, then the flag; pull: everybody else's slice as soon as its flag is up
            const size_t count = (size_t)plan.w[j] * n;
            for (uint32_t i = 0; i < nl; i++) {
                gl_group_rank& rk = g->r[i];
                cudaSetDevice(rk.ctx->device);
                u64* base = hs[i]->coeffs.get() + (size_t)plan.base[j] * n;
                cudaError_t ce = cudaMemcpyAsync(rk.xbuf + xoff[j], base + (size_t)(g->rank0 + i) * count, count * 8,
                                                 cudaMemcpyDeviceToDevice, rk.comm_stream);
                if (ce != cudaSuccess) return gfail(g, GL_E_CUDA, cudaGetErrorString(ce));
                k_group_signal<<<1, 1, 0, rk.comm_stream>>>(rk.xbuf + j, g->epoch);
                ++g_gl_launches;
            }
            for (uint32_t i = 0; i < nl; i++) {
                gl_group_rank& rk = g->r[i];
                cudaSetDevice(rk.ctx->device);
                u64* base = hs[i]->coeffs.get() + (size_t)plan.base[j] * n;
                // 56 CTAs x 256 threads x 4 x 16 B = 0.9 MB of loads in flight per GPU: at 8 GPUs 28 CTAs cost 1.2 ms of a
                // commit, 126 cost 0.3 ms (they crowd the hashing), 56 are the best of the three
                static const unsigned pull_ctas = getenv("GL_B200_GROUP_PULL_CTAS") ? (unsigned)atoi(getenv("GL_B200_GROUP_PULL_CTAS")) : 56u;
                const unsigned per_peer = count >= ((size_t)1 << 18) ? (pull_ctas + G - 2) / (G - 1) : 2u;
                k_group_pull<<<dim3(per_peer, G), 256, 0, rk.comm_stream>>>(rk.d_peer_x, g->rank0 + i, j, g->epoch, xoff[j], base, count);
                ++g_gl_launches;
            }
        } else if (G > 1) {
            if (nl > 1) NCK(g, a->GroupStart());
            for (uint32_t i = 0; i < nl; i++) {
                gl_group_rank& rk = g->r[i];
                cudaSetDevice(rk.ctx->device);
                u64* base = hs[i]->coeffs.get() + (size_t)plan.base[j] * n;
                const size_t count = (size_t)plan.w[j] * n;
                ncclResult_t r = a->AllGather(base + (size_t)(g->rank0 + i) * count, base, count, ncclUint64, rk.comm, rk.comm_stream);
                if (r != ncclSuccess) {
                    if (nl > 1) a->GroupEnd();
                    return gfail(g, GL_E_NCCL, std::string("ncclAllGather: ") + a->GetErrorString(r));
                }
            }
            if (nl > 1) NCK(g, a->GroupEnd());
        }
        for (uint32_t i = 0; i < nl; i++) {
            cudaSetDevice(g->r[i].ctx->device);
            cudaEventRecord(g->r[i].ev[2 * j + 1], g->r[i].comm_stream);
            trace[i].mark("gath" + std::to_string(j), g->r[i].comm_stream);
        }
        if (j > 0)
            for (uint32_t i = 0; i < nl; i++) TRY(lde_round(i, j - 1));
    }
    for (uint32_t i = 0; i < nl; i++) TRY(lde_round(i, plan.rounds - 1));
    // ---- trees, then the cap all-gather on the communication stream
    const uint32_t tail = 2 * plan.rounds;
    for (uint32_t i = 0; i < nl; i++) {
        gl_group_rank& rk = g->r[i];
        gl_ctx* ctx = rk.ctx;
        gl_commit* h = hs[i].get();
        cudaSetDevice(ctx->device);
        h->cols_added = c;
        GTRY(g, ctx, commit_tree(ctx, h, nullptr, GL_DEVICE, h->stream_hash && h->hashed_cols == h->c));
        cudaEventRecord(rk.ev[tail], ctx->stream);
        trace[i].mark("tree", ctx->stream);
        cudaStreamWaitEvent(rk.comm_stream, rk.ev[tail], 0);
    }
    if (G > 1) {
        if (nl > 1) NCK(g, a->GroupStart());
        for (uint32_t i = 0; i < nl; i++) {
            gl_group_rank& rk = g->r[i];
            cudaSetDevice(rk.ctx->device);
            ncclResult_t r = a->AllGather(hs[i]->cap.get(), rk.cap_all, hs[i]->cap.bytes() / 8, ncclUint64, rk.comm, rk.comm_stream);
            if (r != ncclSuccess) {
                if (nl > 1) a->GroupEnd();
                return gfail(g, GL_E_NCCL, std::string("ncclAllGather(cap): ") + a->GetErrorString(r));
            }
        }
        if (nl > 1) NCK(g, a->GroupEnd());
    }
    for (uint32_t i = 0; i < nl; i++) {
        gl_group_rank& rk = g->r[i];
        gl_ctx* ctx = rk.ctx;
        cudaSetDevice(ctx->device);
        if (G == 1) cudaMemcpyAsync(rk.cap_all, hs[i]->cap.get(), cap_bytes, cudaMemcpyDeviceToDevice, rk.comm_stream);
        if (cap_out && cap_out[i])
            cudaMemcpyAsync(cap_out[i], rk.cap_all, cap_bytes, space == GL_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost,
                            rk.comm_stream);
        if (space == GL_DEVICE && coeffs_out && coeffs_out[i])
            cudaMemcpyAsync(coeffs_out[i], hs[i]->coeffs.get(), (size_t)c * n * 8, cudaMemcpyDeviceToDevice, ctx->stream);
    }
    // ---- one host synchronisation per commit
    int rc = GL_OK;
    for (uint32_t i = 0; i < nl; i++) {
        gl_group_rank& rk = g->r[i];
        gl_ctx* ctx = rk.ctx;
        cudaSetDevice(ctx->device);
        cudaError_t e1 = cudaStreamSynchronize(ctx->stream), e2 = cudaStreamSynchronize(rk.comm_stream);
        if (rc == GL_OK && e1 != cudaSuccess) rc = gfail(g, GL_E_CUDA, std::string("commit: ") + cudaGetErrorString(e1));
        if (rc == GL_OK && e2 != cudaSuccess) rc = gfail(g, GL_E_CUDA, std::string("collectives: ") + cudaGetErrorString(e2));
        if (space == GL_HOST) {
            int rc2 = downloads_wait(ctx);
            if (rc == GL_OK && rc2 != GL_OK) rc = gfail(g, rc2, ctx->err);
        }
        trace[i].mark("cap+d2h", rk.comm_stream);
        if (trace[i].on) { cudaStreamSynchronize(rk.comm_stream); trace[i].dump(g->rank0 + i, ctx->ev[0]); }
        if (rc == GL_OK) {
            commit_done(ctx, hs[i].get());
            if (i == 0) memcpy(g->phase_ms, ctx->phase_ms, sizeof g->phase_ms);
        }
    }
    if (rc != GL_OK) return rc;
    for (uint32_t i = 0; i < nl; i++) handles[i] = hs[i].release();
    return GL_OK;
}

extern "C" int gl_group_commit_from_values(gl_group* g, const uint64_t* const* values, uint32_t log_n, uint32_t c,
                                           uint32_t rate_bits, uint32_t cap_height, uint64_t* const* coeffs_out,
                                           uint64_t* const* cap_out, gl_commit** handles, int space, uint32_t flags) {
    return group_commit(g, values, true, log_n, c, rate_bits, cap_height, coeffs_out, cap_out, handles, space, flags,
                        "PolynomialBatch::from_values");
}
extern "C" int gl_group_commit_from_coeffs(gl_group* g, const uint64_t* const* coeffs, uint32_t log_n, uint32_t c,
                                           uint32_t rate_bits, uint32_t cap_height, uint64_t* const* cap_out,
                                           gl_commit** handles, int space, uint32_t flags) {
    return group_commit(g, coeffs, false, log_n, c, rate_bits, cap_height, nullptr, cap_out, handles, space, flags,
                        "PolynomialBatch::from_coeffs");
}

// MerkleTree::get + MerkleTree::prove for k GLOBAL leaf indices of a sharded commit (the FRI query openings,
// fri_prover_query_round): every index is served by the rank that owns the leaf; rows and paths travel over NCCL so
// that EVERY rank ends with all k rows [k][c] and paths [k][L][4].  The exchange is an all-reduce (sum) of a buffer
// in which only the owner of entry q wrote non-zero data: exact for u64, one collective whatever the owner pattern.
extern "C" int gl_group_commit_open(gl_group* g, gl_commit* const* handles, const uint64_t* leaf_indices, uint32_t k,
                                    uint64_t* const* rows_out, uint64_t* const* paths_out, int space) {
    if (!g) return GL_E_ARG;
    if (!handles || (k && !leaf_indices)) return gfail(g, GL_E_ARG, "gl_group_commit_open: NULL argument");
    if (k == 0) return GL_OK;
    if (space != GL_HOST) return gfail(g, GL_E_ARG, "gl_group_commit_open: indices and outputs are host buffers (space = GL_HOST)");
    std::lock_guard<std::mutex> lk(g->mu);
    std::vector<std::unique_lock<std::mutex>> ctx_locks;
    for (auto& rk : g->r) ctx_locks.emplace_back(rk.ctx->mu);
    auto* a = glnccl::api();
    const uint32_t nl = g->nlocal;
    int prev = -1;
    cudaGetDevice(&prev);
    struct Restore { int d; ~Restore() { if (d >= 0) cudaSetDevice(d); } } restore{prev};
    const gl_commit* h0 = handles[0];
    if (!h0) return gfail(g, GL_E_ARG, "gl_group_commit_open: NULL handle");
    const unsigned L = h0->log_n + h0->rate_bits - h0->cap_height;
    const u64 N = (u64)1 << (h0->log_n + h0->rate_bits);
    const size_t row_words = leaf_len(h0), per = row_words + 4 * (size_t)L, words = per * k;
    for (uint32_t q = 0; q < k; q++)
        if (leaf_indices[q] >= N) return gfail(g, GL_E_ARG, "MerkleTree::get / prove: leaf index out of range");
    for (uint32_t i = 0; i < nl; i++) {
        gl_group_rank& rk = g->r[i];
        const gl_commit* h = handles[i];
        if (!h || h->ctx != rk.ctx || !h->finished || h->c != h0->c || h->salt != h0->salt || h->log_n != h0->log_n || h->rate_bits != h0->rate_bits ||
            h->cap_height != h0->cap_height || h->shard_count != g->nranks)
            return gfail(g, GL_E_STATE, "gl_group_commit_open: handles[i] is not this group's shard of one commit");
        gl_ctx* ctx = rk.ctx;
        GCK(g, cudaSetDevice(ctx->device));
        if (rk.open_bytes < words * 8) {
            cudaStreamSynchronize(rk.comm_stream);
            if (rk.open_buf) cudaFree(rk.open_buf);
            rk.open_buf = nullptr;
            GCK(g, cudaMalloc(&rk.open_buf, words * 8));
            rk.open_bytes = words * 8;
        }
        GCK(g, cudaMemsetAsync(rk.open_buf, 0, words * 8, ctx->stream));
        // the indices this rank owns, their slots in the exchange buffer
        std::vector<u64> meta;   // [local index..., slot...]
        std::vector<u64> loc, slot;
        for (uint32_t q = 0; q < k; q++) {
            const u64 v = leaf_indices[q];
            if (v >= h->leaf_begin && v < h->leaf_begin + h->n_local) {
                loc.push_back(v - h->leaf_begin);
                slot.push_back(q);
            }
        }
        const uint32_t mine = (uint32_t)loc.size();
        if (mine) {
            meta = loc;
            meta.insert(meta.end(), slot.begin(), slot.end());
            void* d;
            GTRY(g, ctx, scratch_get(ctx, 3, meta.size() * 8 + 8, &d));
            GCK(g, cudaMemcpyAsync(d, meta.data(), meta.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
            GCK(g, cudaStreamSynchronize(ctx->stream));   // `meta` dies with this iteration
            const u64* d_loc = (const u64*)d;
            const u64* d_slot = d_loc + mine;
            launch_gather_open(h->lde.get(), h->n_local, leaf_len(h), h->digests.get(), L, d_loc, d_slot, mine, rk.open_buf, per, ctx->stream);
        }
        GCK(g, cudaEventRecord(ctx->dl_ev, ctx->stream));
        GCK(g, cudaStreamWaitEvent(rk.comm_stream, ctx->dl_ev, 0));
    }
    if (g->nranks > 1) {
        if (nl > 1) NCK(g, a->GroupStart());
        for (uint32_t i = 0; i < nl; i++) {
            gl_group_rank& rk = g->r[i];
            cudaSetDevice(rk.ctx->device);
            ncclResult_t r = a->AllReduce(rk.open_buf, rk.open_buf, words, ncclUint64, ncclSum, rk.comm, rk.comm_stream);
            if (r != ncclSuccess) {
                if (nl > 1) a->GroupEnd();
                return gfail(g, GL_E_NCCL, std::string("ncclAllReduce(openings): ") + a->GetErrorString(r));
            }
        }
        if (nl > 1) NCK(g, a->GroupEnd());
    }
    std::vector<u64> host(words);
    for (uint32_t i = 0; i < nl; i++) {
        gl_group_rank& rk = g->r[i];
        cudaSetDevice(rk.ctx->device);
        const bool want = (rows_out && rows_out[i]) || (paths_out && paths_out[i]);
        if (want) GCK(g, cudaMemcpyAsync(host.data(), rk.open_buf, words * 8, cudaMemcpyDeviceToHost, rk.comm_stream));
        GCK(g, cudaStreamSynchronize(rk.comm_stream));
        if (!want) continue;
        for (uint32_t q = 0; q < k; q++) {
            if (rows_out && rows_out[i]) memcpy(rows_out[i] + (size_t)q * row_words, host.data() + q * per, row_words * 8);
            if (paths_out && paths_out[i] && L) memcpy(paths_out[i] + (size_t)q * 4 * L, host.data() + q * per + row_words, (size_t)L * 32);
        }
    }
    return GL_OK;
}
