// libgl_b200.so -- the C ABI declared in include/gl_b200.h (host orchestration; kernels live in
// ntt_kernels.cu and hash_kernels.cu).
//
// Device data layout (DESIGN.md section 3):
//   polynomials      [c][n]        column after column (what Vec<PolynomialValues<F>> flattens to)
//   LDE "leaves"     [c][N_local]  COLUMN-major, leaf order along the fast axis: element (leaf i, col j)
//                                  at lde[j * N_local + i].  Leaf order = reverse_index_bits of the
//                                  natural coset order, which is exactly what a decimation-in-frequency
//                                  NTT leaves behind, so "transpose LDEs" + reverse_index_bits_in_place
//                                  of PolynomialBatch::from_coeffs never run as separate passes.
//   digests          [2*(N_local - caps_local)][4]  plonky2's recursive in-order layout
//   cap              [caps_local][4]
// There is no CPU fallback anywhere in this file: every entry point needs a live CUDA context.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <random>
#include <mutex>
#include <new>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/gl_b200.h"
#include "gl_field.cuh"
#include "fri_kernels.h"
#include "hash_kernels.h"
#include "host_staging.h"
#include "ntt_kernels.h"
#include "permutation_kernels.h"
#include "poseidon_constants.h"
#include "quotient_kernels.h"
#include "smt_kernels.h"
#include "smt_proofs.h"

std::atomic<unsigned long long> g_gl_launches{0};

#define GL_PHASES 6  // copy-in, IFFT, coefficients out, LDE NTT, leaf hashing, tree levels

static std::string g_create_error;

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

struct gl_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    uint32_t shard_index = 0, shard_count = 1;
    uint32_t compat = 0;   // GL_COMPAT_*: fork-version switches (gl_ctx_set_compat)
    int tma_shift_tables = 0;   // cached TMA twiddle tables that belong to caller-chosen coset shifts (bounded)
    uint64_t salt_seed = 0, salt_counter = 0;   // blinding salt: seed from the OS at creation (gl_ctx_set_salt_seed overrides)
    std::map<std::tuple<int, uint64_t, uint64_t, uint64_t>, u64*> tables;
    DevBuf scratch[6];
    std::mutex mu;
    // freed commit buffers, kept for the next commit of the same geometry (cudaMalloc/cudaFree of
    // multi-GB blocks cost milliseconds and serialise the device)
    std::multimap<size_t, void*> pool;
    size_t pool_bytes = 0;
    std::map<void*, size_t> user_allocs;   // gl_dev_alloc blocks
    // phase boundaries of the last commit (CUDA events on `stream`)
    cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;   // PCIe copies of the host-buffer commit pipeline
    std::vector<cudaEvent_t> pipe_ev;
    staging::Ring h2d_ring;                 // page-able caller memory goes through these (host_staging.h)
    staging::Downloader* downloader = nullptr;
    cudaEvent_t dl_ev = nullptr;
    cudaEvent_t ev[GL_PHASES + 1] = {};
    bool ev_valid = false;
    float phase_ms[GL_PHASES] = {};
};

static int fail(gl_ctx* ctx, int code, const std::string& msg) {
    if (ctx) ctx->err = msg;
    else g_create_error = msg;
    return code;
}
static int cuda_fail(gl_ctx* ctx, cudaError_t e, const char* what) {
    std::string msg = std::string(what) + ": " + cudaGetErrorString(e);
    cudaGetLastError();
    return fail(ctx, e == cudaErrorMemoryAllocation ? GL_E_OOM : GL_E_CUDA, msg);
}
#define CK(call)                                                   \
    do {                                                           \
        cudaError_t e__ = (call);                                  \
        if (e__ != cudaSuccess) return cuda_fail(ctx, e__, #call); \
    } while (0)
#define TRY(expr)             \
    do {                      \
        int rc__ = (expr);    \
        if (rc__) return rc__; \
    } while (0)

static inline unsigned ilog2(uint64_t x) { return 63u - (unsigned)__builtin_clzll(x); }
static inline bool is_pow2(uint64_t x) { return x && !(x & (x - 1)); }
static inline uint64_t bitrev(uint64_t x, unsigned bits) {
    uint64_t r = 0;
    for (unsigned i = 0; i < bits; i++) r |= ((x >> i) & 1) << (bits - 1 - i);
    return r;
}

struct Guard {  // binds the ctx's device for the duration of a call and serialises calls on one ctx
    std::unique_lock<std::mutex> lk;
    int prev = -1;
    explicit Guard(gl_ctx* ctx) : lk(ctx->mu) {
        cudaGetDevice(&prev);
        if (prev != ctx->device) cudaSetDevice(ctx->device);
        else prev = -1;
    }
    ~Guard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

static int scratch_get(gl_ctx* ctx, int slot, size_t bytes, void** out) {
    *out = nullptr;
    DevBuf& b = ctx->scratch[slot];
    if (b.cap < bytes) {
        if (b.p) {
            CK(cudaStreamSynchronize(ctx->stream));
            cudaFree(b.p);
            b.p = nullptr;
            b.cap = 0;
        }
        size_t want = bytes + bytes / 8;
        cudaError_t e = cudaMalloc(&b.p, want);
        if (e != cudaSuccess) {
            cudaGetLastError();
            want = bytes;
            e = cudaMalloc(&b.p, want);
        }
        if (e != cudaSuccess) return cuda_fail(ctx, e, "cudaMalloc(scratch)");
        b.cap = want;
    }
    *out = b.p;
    return GL_OK;
}

static void pool_trim(gl_ctx* ctx) {
    for (auto& kv : ctx->pool) cudaFree(kv.second);
    ctx->pool.clear();
    ctx->pool_bytes = 0;
}
static int dev_alloc(gl_ctx* ctx, size_t bytes, u64** out) {
    void* p = nullptr;
    if (bytes == 0) bytes = 8;
    auto it = ctx->pool.find(bytes);
    if (it != ctx->pool.end()) {
        *out = (u64*)it->second;
        ctx->pool.erase(it);
        ctx->pool_bytes -= bytes;
        return GL_OK;
    }
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaErrorMemoryAllocation && !ctx->pool.empty()) {
        cudaGetLastError();
        cudaStreamSynchronize(ctx->stream);
        pool_trim(ctx);
        e = cudaMalloc(&p, bytes);
    }
    if (e != cudaSuccess) return cuda_fail(ctx, e, "cudaMalloc");
    *out = (u64*)p;
    return GL_OK;
}
// stream-ordered reuse: every consumer of a pooled block runs on ctx->stream
static void dev_release(gl_ctx* ctx, void* p, size_t bytes) {
    if (!p) return;
    if (bytes == 0) bytes = 8;
    if (ctx->pool_bytes + bytes > ((size_t)48 << 30)) {
        cudaFree(p);
        return;
    }
    ctx->pool.emplace(bytes, p);
    ctx->pool_bytes += bytes;
}

// The one owner of a pooled block: the block goes back to the pool when the owner is reset or dies.  An owner dies
// with the ctx's mutex held and its device current (declare it after the Guard).
class PoolBuf {
  public:
    PoolBuf() = default;
    PoolBuf(const PoolBuf&) = delete;
    PoolBuf& operator=(const PoolBuf&) = delete;
    PoolBuf(PoolBuf&& o) noexcept : ctx_(o.ctx_), p_(o.p_), bytes_(o.bytes_) { o.p_ = nullptr; }
    PoolBuf& operator=(PoolBuf&& o) noexcept {
        if (this != &o) {
            reset();
            ctx_ = o.ctx_;
            p_ = o.p_;
            bytes_ = o.bytes_;
            o.p_ = nullptr;
        }
        return *this;
    }
    ~PoolBuf() { reset(); }
    int alloc(gl_ctx* ctx, size_t bytes) {
        reset();
        TRY(dev_alloc(ctx, bytes, &p_));
        ctx_ = ctx;
        bytes_ = bytes;
        return GL_OK;
    }
    void reset() {
        dev_release(ctx_, p_, bytes_);
        p_ = nullptr;
    }
    u64* get() const { return p_; }
    size_t bytes() const { return bytes_; }

  private:
    gl_ctx* ctx_ = nullptr;
    u64* p_ = nullptr;
    size_t bytes_ = 0;
};

struct gl_commit {
    gl_ctx* ctx = nullptr;
    uint32_t log_n = 0, c = 0, rate_bits = 0, cap_height = 0;
    uint32_t salt = 0;         // blinding: SALT_SIZE = 4 random columns after the c polynomial columns of every leaf
    uint32_t shard_index = 0, shard_count = 1;
    uint64_t n_local = 0;      // leaves held here
    uint64_t leaf_begin = 0;   // global index of the first local leaf
    uint32_t cap_local_bits = 0;
    PoolBuf coeffs;            // [c][n]
    PoolBuf lde;               // [c + salt][n_local]
    PoolBuf digests;           // [2*(n_local - 2^cap_local_bits)][4]
    PoolBuf cap;               // [2^cap_local_bits][4]
    uint64_t num_digests = 0;
    uint32_t cols_added = 0;   // gl_commit_begin / add_coeffs / finish
    bool finished = true;
    // GL_COMMIT_STREAM_HASH: leaves are absorbed 8 polynomials at a time as the blocks arrive
    bool stream_hash = false;
    uint32_t next_col = 0, hashed_cols = 0;
    PoolBuf hstate;            // [12][n_local] sponge states between blocks
};

static inline uint32_t leaf_len(const gl_commit* h) { return h->c + h->salt; }   // MerkleTree.leaves[i].len()

// Host <-> device copies of caller buffers.  Page-able memory of a megabyte or more is staged through
// page-locked rings by helper threads (host_staging.h); small or page-locked buffers go straight to the DMA engine.
static size_t staged_min_bytes() {   // GL_B200_STAGING=0 hands page-able memory to the driver instead (A/B measurements)
    static const size_t v = [] {
        const char* e = getenv("GL_B200_STAGING");
        return (e && e[0] == '0') ? ~(size_t)0 : (size_t)1 << 20;
    }();
    return v;
}
#define STAGED_MIN_BYTES staged_min_bytes()
static int h2d_copy(gl_ctx* ctx, void* ddst, const staging::HostSeg* segs, size_t count, cudaStream_t stream) {
    size_t total = 0;
    for (size_t i = 0; i < count; i++) total += segs[i].bytes;
    if (total < STAGED_MIN_BYTES) {
        char* to = (char*)ddst;
        for (size_t i = 0; i < count; i++) {
            if (segs[i].bytes) CK(cudaMemcpyAsync(to, segs[i].ptr, segs[i].bytes, cudaMemcpyHostToDevice, stream));
            to += segs[i].bytes;
        }
        return GL_OK;
    }
    CK(staging::h2d_gather(ctx->h2d_ring, ddst, segs, count, stream));
    return GL_OK;
}
static int h2d_copy(gl_ctx* ctx, void* ddst, const void* src, size_t bytes, cudaStream_t stream) {
    if (bytes < STAGED_MIN_BYTES) {
        if (bytes) CK(cudaMemcpyAsync(ddst, src, bytes, cudaMemcpyHostToDevice, stream));
        return GL_OK;
    }
    staging::HostSeg seg{const_cast<void*>(src), bytes};
    return h2d_copy(ctx, ddst, &seg, 1, stream);
}
// `ready`: an event already recorded after the producer of dsrc; the copy runs on d2h_stream (or its worker)
// and is complete after downloads_wait().
static int d2h_copy(gl_ctx* ctx, std::vector<staging::HostSeg> segs, const void* dsrc, cudaEvent_t ready) {
    size_t total = 0;
    bool pinned = true;
    for (auto& sg : segs) {
        total += sg.bytes;
        if (pinned && sg.bytes) pinned = staging::is_pinned(sg.ptr);
    }
    if (!total) return GL_OK;
    if (pinned || total < STAGED_MIN_BYTES) {
        CK(cudaStreamWaitEvent(ctx->d2h_stream, ready, 0));
        const char* from = (const char*)dsrc;
        for (auto& sg : segs) {
            if (sg.bytes) CK(cudaMemcpyAsync(sg.ptr, from, sg.bytes, cudaMemcpyDeviceToHost, ctx->d2h_stream));
            from += sg.bytes;
        }
        return GL_OK;
    }
    if (!ctx->downloader) {
        ctx->downloader = new (std::nothrow) staging::Downloader(ctx->device, ctx->d2h_stream);
        if (!ctx->downloader) return fail(ctx, GL_E_OOM, "host allocation failed");
    }
    ctx->downloader->submit(dsrc, std::move(segs), ready);
    return GL_OK;
}
static int downloads_wait(gl_ctx* ctx) {
    cudaError_t e = cudaSuccess;
    if (ctx->downloader) e = ctx->downloader->wait();
    cudaError_t e2 = cudaStreamSynchronize(ctx->d2h_stream);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "download to host memory");
    if (e2 != cudaSuccess) return cuda_fail(ctx, e2, "download to host memory");
    return GL_OK;
}

// A GL_DEVICE buffer goes to the kernels as it is, and they read and write it in 16-byte pairs (Poseidon states,
// digests, NTT outputs) or through TMA descriptors, whose base must be 16-byte aligned.  So a device buffer of 16 bytes
// or more must be 16-byte aligned, a smaller one 8-byte aligned; GL_E_ARG otherwise, before any copy or launch.
// Host buffers are staged into pool blocks and need nothing.  `what` names the entry point and the argument.
static int check_device_ptr(gl_ctx* ctx, int space, const void* p, size_t bytes, const char* what) {
    if (space != GL_DEVICE || !p || !bytes) return GL_OK;
    const uintptr_t align = bytes >= 16 ? 16 : 8;
    if (((uintptr_t)p & (align - 1)) == 0) return GL_OK;
    return fail(ctx, GL_E_ARG, std::string(what) + ": GL_DEVICE buffer is not " + std::to_string(align) +
                                   "-byte aligned (device buffers of 16 bytes or more need 16-byte alignment)");
}

// caller buffer -> device pointer (no copy when the caller already is on the device)
static int stage_in(gl_ctx* ctx, const void* src, size_t bytes, int space, int slot, const u64** out) {
    if (space == GL_DEVICE) {
        *out = (const u64*)src;
        return GL_OK;
    }
    void* d;
    TRY(scratch_get(ctx, slot, bytes ? bytes : 8, &d));
    TRY(h2d_copy(ctx, d, src, bytes, ctx->stream));
    *out = (const u64*)d;
    return GL_OK;
}
static int copy_out(gl_ctx* ctx, void* dst, const void* dsrc, size_t bytes, int space) {
    if (!dst || !bytes || dst == dsrc) return GL_OK;
    if (space == GL_HOST && bytes >= STAGED_MIN_BYTES && !staging::is_pinned(dst)) {
        // Callers reuse or free `dsrc` right after this returns (stream order covered that when the copy was a
        // cudaMemcpyAsync on ctx->stream), so the staged download completes before we go on.
        CK(cudaEventRecord(ctx->dl_ev, ctx->stream));
        TRY(d2h_copy(ctx, {staging::HostSeg{dst, bytes}}, dsrc, ctx->dl_ev));
        return downloads_wait(ctx);
    }
    CK(cudaMemcpyAsync(dst, dsrc, bytes, space == GL_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost,
                       ctx->stream));
    return GL_OK;
}
static int finish(gl_ctx* ctx) {
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->stream));
    return GL_OK;
}

// ------------------------------------------------------------------------------------------------
// tables (built on the host with exact 128-bit arithmetic, cached on the device)
// ------------------------------------------------------------------------------------------------
enum { TAB_SMALL = 1, TAB_POW = 2, TAB_COSETS = 3, TAB_FULL = 4, TAB_DIRECT = 5, TAB_COSETS_DIRECT = 6, TAB_TMA_POST = 7 };

static void fill_pow_table(u64* t, u64 base) {  // [3][1024]: base^e, base^(1024 e), base^(2^20 e)
    u64 b = glh::canon(base);
    for (int lvl = 0; lvl < 3; lvl++) {
        u64 acc = 1;
        for (int e = 0; e < 1024; e++) {
            t[lvl * 1024 + e] = acc;
            acc = glh::mul(acc, b);
        }
        b = acc;  // base^(1024)
    }
}

static int table_upload(gl_ctx* ctx, std::tuple<int, uint64_t, uint64_t, uint64_t> key, const std::vector<u64>& host,
                        const u64** out) {
    u64* d;
    TRY(dev_alloc(ctx, host.size() * sizeof(u64), &d));
    CK(cudaMemcpyAsync(d, host.data(), host.size() * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));  // `host` dies with the caller
    ctx->tables[key] = d;
    *out = d;
    return GL_OK;
}

// w_{2^m}^x for x < 2^(m-1)  (inverse: w^-x)
static int small_table(gl_ctx* ctx, unsigned m, bool inverse, const u64** out) {
    auto key = std::make_tuple((int)TAB_SMALL, (uint64_t)m, (uint64_t)inverse, (uint64_t)0);
    auto it = ctx->tables.find(key);
    if (it != ctx->tables.end()) {
        *out = it->second;
        return GL_OK;
    }
    size_t len = m ? ((size_t)1 << (m - 1)) : 1;
    std::vector<u64> h(len);
    u64 w = glh::root_of_unity(m);
    if (inverse) w = glh::inv(w);
    u64 acc = 1;
    for (size_t i = 0; i < len; i++) {
        h[i] = acc;
        acc = glh::mul(acc, w);
    }
    return table_upload(ctx, key, h, out);
}

static int pow_table(gl_ctx* ctx, u64 base, const u64** out) {
    auto key = std::make_tuple((int)TAB_POW, (uint64_t)glh::canon(base), (uint64_t)0, (uint64_t)0);
    auto it = ctx->tables.find(key);
    if (it != ctx->tables.end()) {
        *out = it->second;
        return GL_OK;
    }
    std::vector<u64> h(3072);
    fill_pow_table(h.data(), base);
    return table_upload(ctx, key, h, out);
}

// one pow table per local leaf block b: shift_b = 7 * w_N^k, k = bitrev_r(global block)
static int coset_tables(gl_ctx* ctx, unsigned lg_n, unsigned r, uint32_t shard_index, uint32_t shard_count,
                        const u64** out) {
    auto key = std::make_tuple((int)TAB_COSETS, (uint64_t)lg_n, (uint64_t)r,
                               ((uint64_t)shard_index << 32) | shard_count);
    auto it = ctx->tables.find(key);
    if (it != ctx->tables.end()) {
        *out = it->second;
        return GL_OK;
    }
    uint32_t blocks = (1u << r) / shard_count;
    std::vector<u64> h((size_t)blocks * 3072);
    u64 wN = glh::root_of_unity(lg_n + r);
    for (uint32_t b = 0; b < blocks; b++) {
        uint64_t k = bitrev((uint64_t)shard_index * blocks + b, r);
        u64 shift = glh::mul(7, glh::pow(wN, k));
        fill_pow_table(h.data() + (size_t)b * 3072, shift);
    }
    return table_upload(ctx, key, h, out);
}

// ------------------------------------------------------------------------------------------------
// NTT driver: natural order in, bit-reversed order out (decimation in frequency), 1..3 passes
// ------------------------------------------------------------------------------------------------
struct NttJob {
    const u64* in = nullptr;
    u64 in_ld = 0, in_coset_stride = 0;
    u64* out = nullptr;
    u64 out_ld = 0, out_coset_stride = 0;
    unsigned L = 0;
    uint32_t columns = 1, cosets = 1;
    bool inverse = false;
    const u64* pre_tab = nullptr;
    bool pre_direct_ok = false;   // pre_tab is the head of a cached coset_tables() block (stable key for the expanded copy)
    u64 final_scale = 1;
    int canonical_out = 0;
};

// w_{2^m}^e for e < 2^m (inverse: w^-e): twiddle table of the fast pass
static int full_table(gl_ctx* ctx, unsigned m, bool inverse, const u64** out) {
    auto key = std::make_tuple((int)TAB_FULL, (uint64_t)m, (uint64_t)inverse, (uint64_t)0);
    auto it = ctx->tables.find(key);
    if (it != ctx->tables.end()) {
        *out = it->second;
        return GL_OK;
    }
    std::vector<u64> h((size_t)1 << m);
    u64 w = glh::root_of_unity(m);
    if (inverse) w = glh::inv(w);
    u64 acc = 1;
    for (auto& v : h) {
        v = acc;
        acc = glh::mul(acc, w);
    }
    return table_upload(ctx, key, h, out);
}

// base^i for i < 2^lg, expanded on the device from the 3 x 1024 power table `pow` (key = the table's pointer)
static int direct_table(gl_ctx* ctx, const u64* pow, unsigned lg, const u64** out) {
    auto key = std::make_tuple((int)TAB_DIRECT, (uint64_t)(uintptr_t)pow, (uint64_t)lg, (uint64_t)0);
    auto it = ctx->tables.find(key);
    if (it != ctx->tables.end()) {
        *out = it->second;
        return GL_OK;
    }
    u64* d;
    TRY(dev_alloc(ctx, sizeof(u64) << lg, &d));
    launch_fill_powers(d, (u64)1 << lg, pow, ctx->stream);
    ctx->tables[key] = d;
    *out = d;
    return GL_OK;
}
// [blocks][2^lg]: shift_b^i for every local coset block b (expanded from coset_tables' power tables)
static int coset_direct_tables(gl_ctx* ctx, const u64* coset_pow, unsigned lg, uint32_t blocks, const u64** out) {
    auto key = std::make_tuple((int)TAB_COSETS_DIRECT, (uint64_t)(uintptr_t)coset_pow, (uint64_t)lg, (uint64_t)blocks);
    auto it = ctx->tables.find(key);
    if (it != ctx->tables.end()) {
        *out = it->second;
        return GL_OK;
    }
    u64* d;
    TRY(dev_alloc(ctx, ((size_t)blocks * sizeof(u64)) << lg, &d));
    for (uint32_t b = 0; b < blocks; b++)
        launch_fill_powers(d + ((size_t)b << lg), (u64)1 << lg, coset_pow + (size_t)b * 3072, ctx->stream);
    ctx->tables[key] = d;
    *out = d;
    return GL_OK;
}

// split of a size-2^L transform into passes; fast[i] says the radix-16 register kernel (m = 8..10) runs it
static unsigned plan_passes(unsigned L, unsigned ms[4], bool fast[4]) {
    auto set = [&](unsigned i, unsigned m, bool f) { ms[i] = m; fast[i] = f; };
    if (L <= 7) { set(0, L, false); return 1; }
    if (L <= 10) { set(0, L, true); return 1; }
    if (L <= 15) { set(0, 8, true); set(1, L - 8, false); return 2; }
    if (L <= 20) { set(0, (L + 1) / 2, true); set(1, L / 2, true); return 2; }
    if (L <= 23) { set(0, 8, true); set(1, 8, true); set(2, L - 16, false); return 3; }
    for (unsigned i = 0; i < 3; i++) set(i, L / 3 + (i < L % 3 ? 1 : 0), true);
    return 3;
}

static bool tma_table_cached(gl_ctx* ctx, const NttJob& j) {
    auto key = std::make_tuple((int)TAB_TMA_POST, (uint64_t)(uintptr_t)j.pre_tab, ((uint64_t)j.L << 1) | (uint64_t)j.inverse,
                               (uint64_t)j.cosets);
    return ctx->tables.find(key) != ctx->tables.end();
}
// tables of the TMA path: post3 [cosets][256][2^s] followed by rowfac [cosets][256] (see ntt_kernels.h)
static int tma_tables(gl_ctx* ctx, const NttJob& j, const u64* post_tab, const u64** post3, const u64** rowfac) {
    const unsigned s = j.L - 8;
    auto key = std::make_tuple((int)TAB_TMA_POST, (uint64_t)(uintptr_t)j.pre_tab, ((uint64_t)j.L << 1) | (uint64_t)j.inverse,
                               (uint64_t)j.cosets);
    const size_t t_elems = ((size_t)j.cosets << 8) << s;
    auto it = ctx->tables.find(key);
    u64* d;
    if (it != ctx->tables.end()) {
        d = const_cast<u64*>(it->second);
    } else {
        TRY(dev_alloc(ctx, (t_elems + (size_t)j.cosets * 256) * sizeof(u64), &d));
        launch_ntt_tma_tables(d, d + t_elems, post_tab, j.pre_tab, s, j.cosets, ctx->stream);
        ctx->tables[key] = d;
        if (j.pre_tab && !j.pre_direct_ok) ctx->tma_shift_tables++;
    }
    *post3 = d;
    *rowfac = j.pre_tab ? d + t_elems : nullptr;
    return GL_OK;
}

static int run_dif(gl_ctx* ctx, const NttJob& j) {
    if (j.columns == 0) return GL_OK;
    const u64 n = (u64)1 << j.L;
    static const bool tma_off = getenv("GL_B200_NTT_TMA") && atoi(getenv("GL_B200_NTT_TMA")) == 0;
    // a caller-chosen coset shift gets its own 2^L-entry table: fine for the handful a prover uses (7, 7^-1, FRI shifts), so
    // the cache takes at most 24 of them and later shifts run on the radix-16 kernels below
    const bool tma_tables_ok = !j.pre_tab || j.pre_direct_ok || tma_table_cached(ctx, j) || ctx->tma_shift_tables < 24;
    if (!tma_off && ntt_tma_supported(j.L) && j.final_scale == 1 && tma_tables_ok &&
        (j.cosets == 1 || (j.in_coset_stride == 0 && j.out_coset_stride == n))) {   // the LDE's geometry: one input, blocks of n out
        u64 w = glh::root_of_unity(j.L);
        if (j.inverse) w = glh::inv(w);
        const u64* post;
        TRY(pow_table(ctx, w, &post));
        ntt_tma_job t;
        memset(&t, 0, sizeof t);
        t.in = j.in; t.in_ld = j.in_ld; t.in_coset_stride = j.in_coset_stride;
        t.out = j.out; t.out_ld = j.out_ld; t.out_coset_stride = j.out_coset_stride;
        t.L = j.L; t.columns = j.columns; t.cosets = j.cosets; t.inverse = j.inverse;
        t.canonical_out = j.canonical_out;
        TRY(full_table(ctx, 8, j.inverse, &t.wt1));
        TRY(full_table(ctx, j.L - 8, j.inverse, &t.wt2));
        TRY(tma_tables(ctx, j, post, &t.post3, &t.rowfac));
        if (launch_ntt_tma(t, ctx->stream)) return GL_OK;
        return fail(ctx, GL_E_CUDA, "ntt: TMA pass launch failed");
    }
    unsigned ms[4];
    bool fast[4];
    const unsigned np = plan_passes(j.L, ms, fast);
    unsigned done = 0;
    for (unsigned i = 0; i < np; i++) {
        const unsigned m = ms[i];
        done += m;
        const unsigned s = j.L - done;
        const bool first = i == 0, last = i == np - 1;
        const u64* post = nullptr;
        if (s) {
            u64 w = glh::root_of_unity(s + m);
            if (j.inverse) w = glh::inv(w);
            TRY(pow_table(ctx, w, &post));
        }
        if (fast[i] && (!last || j.final_scale == 1)) {
            ntt16_args f;
            memset(&f, 0, sizeof f);
            f.in = first ? j.in : j.out;
            f.in_ld = first ? j.in_ld : j.out_ld;
            f.in_coset_stride = first ? j.in_coset_stride : j.out_coset_stride;
            f.out = j.out; f.out_ld = j.out_ld; f.out_coset_stride = j.out_coset_stride;
            f.pre_tab = first ? j.pre_tab : nullptr;
            f.post_tab = post;
            // large transforms: one table load instead of two lookups and a multiply per element
            if (j.L >= 16 && j.L <= 22 && j.columns >= 8) {
                if (post && s + m <= 22) TRY(direct_table(ctx, post, s + m, &f.post_direct));
                if (f.pre_tab && j.pre_direct_ok) TRY(coset_direct_tables(ctx, j.pre_tab, j.L, j.cosets, &f.pre_direct));
            }
            TRY(full_table(ctx, m, j.inverse, &f.wtab));
            f.s = s;
            f.canonical_out = last ? j.canonical_out : 0;
            if (launch_ntt16(f, m, j.inverse, n, j.columns, j.cosets, ctx->stream)) continue;
        }
        ntt_pass_args a;
        memset(&a, 0, sizeof a);
        a.m = m;
        a.s = s;
        a.in = first ? j.in : j.out;
        a.in_ld = first ? j.in_ld : j.out_ld;
        a.in_coset_stride = first ? j.in_coset_stride : j.out_coset_stride;
        a.out = j.out;
        a.out_ld = j.out_ld;
        a.out_coset_stride = j.out_coset_stride;
        a.pre_tab = first ? j.pre_tab : nullptr;
        TRY(small_table(ctx, a.m, j.inverse, &a.small_tab));
        if (a.s) {
            a.post_tab = post;
            a.T = a.s >= 3 ? 8 : (1u << a.s);
            a.rows = (u64)1 << a.m;
        } else {
            a.post_tab = nullptr;
            a.T = 1;
            u64 blk = (u64)1 << a.m;
            a.rows = n < 4096 ? n : 4096;
            if (a.rows < blk) a.rows = blk;
        }
        a.final_scale = last ? j.final_scale : 1;
        a.canonical_out = last ? j.canonical_out : 0;
        launch_ntt_pass(a, n, j.columns, j.cosets, ctx->stream);
    }
    return GL_OK;
}

// natural -> natural transform of [c][n] columns at `data` (device), through scratch slot 1
// `src` (default: data itself) holds the input columns; the result always lands in `data`
static int transform_natural(gl_ctx* ctx, u64* data, unsigned L, uint32_t c, bool inverse, const u64* pre_tab,
                             const u64* post_scale_tab, const u64* src = nullptr) {
    const u64 n = (u64)1 << L;
    void* tmp;
    TRY(scratch_get(ctx, 1, (size_t)c * n * sizeof(u64), &tmp));
    NttJob j;
    j.in = src ? src : data; j.in_ld = n; j.out = (u64*)tmp; j.out_ld = n;
    j.L = L; j.columns = c; j.cosets = 1; j.inverse = inverse; j.pre_tab = pre_tab;
    TRY(run_dif(ctx, j));
    u64 scale = inverse ? glh::inv(glh::canon(n % GL_P)) : 1;
    launch_bitrev_permute((const u64*)tmp, n, data, n, L, c, scale, ctx->stream);
    if (post_scale_tab) launch_scale_powers(data, n, n, c, post_scale_tab, ctx->stream);
    return GL_OK;
}

// ------------------------------------------------------------------------------------------------
// context API
// ------------------------------------------------------------------------------------------------
extern "C" int gl_ctx_create(int device, gl_ctx** out) {
    if (!out) return fail(nullptr, GL_E_ARG, "gl_ctx_create: out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(nullptr, GL_E_CUDA,
                    std::string("gl_ctx_create: no CUDA device (this library has no CPU fallback): ") +
                        cudaGetErrorString(e));
    }
    if (device < 0 || device >= count) return fail(nullptr, GL_E_ARG, "gl_ctx_create: bad device index");
    gl_ctx* ctx = new (std::nothrow) gl_ctx();
    if (!ctx) return fail(nullptr, GL_E_OOM, "gl_ctx_create: host allocation failed");
    ctx->device = device;
    int prev = -1;
    cudaGetDevice(&prev);
    e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->h2d_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        int rc = cuda_fail(nullptr, e, "gl_ctx_create");
        gl_ctx_destroy(ctx);
        return rc;
    }
    for (auto& ev : ctx->ev) cudaEventCreate(&ev);
    cudaEventCreateWithFlags(&ctx->dl_ev, cudaEventDisableTiming);
    uint64_t rc360[360];
    if (!poseidon_constants::generate(rc360)) {
        gl_ctx_destroy(ctx);
        return fail(nullptr, GL_E_STATE, "gl_ctx_create: derived Poseidon round constants fail their fingerprint");
    }
    int up = gl_poseidon_upload_constants(rc360);
    if (up != 0) {
        int rc = cuda_fail(nullptr, (cudaError_t)up, "upload Poseidon constants");
        gl_ctx_destroy(ctx);
        return rc;
    }
    int st = gl_field_selftest(ctx->stream);
    if (st != 0) {
        int rc = st < 0 ? cuda_fail(nullptr, (cudaError_t)(-st), "field self-test")
                        : fail(nullptr, GL_E_STATE, "gl_ctx_create: Goldilocks add/sub/mul self-test failed on this device/toolchain (pair " +
                                                        std::to_string(st - 1) + ")");
        gl_ctx_destroy(ctx);
        return rc;
    }
    {   // salt seed for blinded commits: the OS entropy source (upstream: F::rand_vec on the thread RNG)
        std::random_device rd;
        ctx->salt_seed = ((uint64_t)rd() << 32) ^ (uint64_t)rd() ^ ((uint64_t)(uintptr_t)ctx << 7);
    }
    if (prev >= 0 && prev != device) cudaSetDevice(prev);
    *out = ctx;
    return GL_OK;
}

extern "C" void gl_ctx_destroy(gl_ctx* ctx) {
    if (!ctx) return;
    {
        Guard g(ctx);
        if (ctx->stream) cudaStreamSynchronize(ctx->stream);
        delete ctx->downloader;   // joins the worker
        ctx->h2d_ring.destroy();
        if (ctx->dl_ev) cudaEventDestroy(ctx->dl_ev);
        for (auto& kv : ctx->tables) cudaFree(kv.second);
        for (auto& b : ctx->scratch)
            if (b.p) cudaFree(b.p);
        for (auto& kv : ctx->user_allocs) cudaFree(kv.first);
        pool_trim(ctx);
        for (auto& ev : ctx->ev)
            if (ev) cudaEventDestroy(ev);
        for (auto& ev : ctx->pipe_ev) cudaEventDestroy(ev);
        if (ctx->h2d_stream) cudaStreamDestroy(ctx->h2d_stream);
        if (ctx->d2h_stream) cudaStreamDestroy(ctx->d2h_stream);
        if (ctx->stream) cudaStreamDestroy(ctx->stream);
    }
    delete ctx;
}

extern "C" const char* gl_last_error(const gl_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }
extern "C" void* gl_ctx_stream(gl_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
extern "C" int gl_ctx_sync(gl_ctx* ctx) {
    if (!ctx) return GL_E_ARG;
    Guard g(ctx);
    return finish(ctx);
}
extern "C" int gl_ctx_set_shard(gl_ctx* ctx, uint32_t index, uint32_t count) {
    if (!ctx) return GL_E_ARG;
    if (!is_pow2(count) || index >= count) return fail(ctx, GL_E_ARG, "gl_ctx_set_shard: count must be a power of two and index < count");
    ctx->shard_index = index;
    ctx->shard_count = count;
    return GL_OK;
}
extern "C" uint64_t gl_ctx_kernel_launches(const gl_ctx*) { return g_gl_launches.load(); }

extern "C" int gl_ctx_commit_phase_ms(const gl_ctx* ctx, float* out6) {
    if (!ctx || !out6 || !ctx->ev_valid) return GL_E_STATE;
    for (int i = 0; i < GL_PHASES; i++) out6[i] = ctx->phase_ms[i];
    return GL_OK;
}
extern "C" int gl_ctx_trim(gl_ctx* ctx) {
    if (!ctx) return GL_E_ARG;
    Guard g(ctx);
    CK(cudaStreamSynchronize(ctx->stream));
    pool_trim(ctx);
    return GL_OK;
}

extern "C" int gl_dev_alloc(gl_ctx* ctx, size_t bytes, void** out) {
    if (!ctx || !out) return GL_E_ARG;
    Guard g(ctx);
    u64* p;
    TRY(dev_alloc(ctx, bytes, &p));
    ctx->user_allocs[p] = bytes ? bytes : 8;
    *out = p;
    return GL_OK;
}
extern "C" void gl_dev_free(gl_ctx* ctx, void* p) {
    if (!ctx || !p) return;
    Guard g(ctx);
    auto it = ctx->user_allocs.find(p);
    if (it == ctx->user_allocs.end()) return;
    cudaStreamSynchronize(ctx->stream);
    dev_release(ctx, p, it->second);
    ctx->user_allocs.erase(it);
}
extern "C" int gl_copy(gl_ctx* ctx, void* dst, int dst_space, const void* src, int src_space, size_t bytes) {
    if (!ctx) return GL_E_ARG;
    if (bytes && (!dst || !src)) return fail(ctx, GL_E_ARG, "gl_copy: NULL buffer");
    Guard g(ctx);
    cudaMemcpyKind kind = dst_space == GL_DEVICE ? (src_space == GL_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice)
                                                 : (src_space == GL_DEVICE ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost);
    if (kind == cudaMemcpyHostToDevice) TRY(h2d_copy(ctx, dst, src, bytes, ctx->stream));
    else if (kind == cudaMemcpyDeviceToHost) TRY(copy_out(ctx, dst, src, bytes, GL_HOST));
    else if (bytes) CK(cudaMemcpyAsync(dst, src, bytes, kind, ctx->stream));
    return finish(ctx);
}

extern "C" int gl_host_alloc(size_t bytes, void** out) {
    if (!out) return GL_E_ARG;
    cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 8, cudaHostAllocPortable);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *out = nullptr;
        return fail(nullptr, GL_E_OOM, std::string("gl_host_alloc: ") + cudaGetErrorString(e));
    }
    return GL_OK;
}
extern "C" void gl_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

// ------------------------------------------------------------------------------------------------
// Poseidon batches
// ------------------------------------------------------------------------------------------------
extern "C" int gl_poseidon_permute_batch(gl_ctx* ctx, uint64_t* states, uint64_t m, int space) {
    if (!ctx) return GL_E_ARG;
    if (m && !states) return fail(ctx, GL_E_ARG, "gl_poseidon_permute_batch: NULL states");
    TRY(check_device_ptr(ctx, space, states, m * 96, "gl_poseidon_permute_batch: states"));
    Guard g(ctx);
    const u64* d;
    TRY(stage_in(ctx, states, m * 96, space, 0, &d));
    launch_permute_batch((u64*)d, m, ctx->stream);
    TRY(copy_out(ctx, states, d, m * 96, space));
    return finish(ctx);
}

extern "C" int gl_poseidon_duplex_chain(gl_ctx* ctx, uint64_t* state, const uint64_t* chunks, uint64_t m) {
    if (!ctx) return GL_E_ARG;
    if (!state || (m && !chunks)) return fail(ctx, GL_E_ARG, "gl_poseidon_duplex_chain: NULL argument");
    if (m > ((uint64_t)1 << 24)) return fail(ctx, GL_E_ARG, "gl_poseidon_duplex_chain: chain too long");
    if (m == 0) return GL_OK;
    Guard g(ctx);
    void* d;
    TRY(scratch_get(ctx, 0, 96 + m * 64, &d));
    u64* dstate = (u64*)d;
    CK(cudaMemcpyAsync(dstate, state, 96, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dstate + 12, chunks, m * 64, cudaMemcpyHostToDevice, ctx->stream));
    launch_duplex_chain(dstate, dstate + 12, m, ctx->stream);
    CK(cudaMemcpyAsync(state, dstate, 96, cudaMemcpyDeviceToHost, ctx->stream));
    return finish(ctx);
}

extern "C" int gl_poseidon_two_to_one_batch(gl_ctx* ctx, const uint64_t* l, const uint64_t* r, uint64_t* out,
                                            uint64_t m, int space) {
    if (!ctx) return GL_E_ARG;
    if (m && (!l || !r || !out)) return fail(ctx, GL_E_ARG, "gl_poseidon_two_to_one_batch: NULL buffer");
    TRY(check_device_ptr(ctx, space, l, m * 32, "gl_poseidon_two_to_one_batch: l"));
    TRY(check_device_ptr(ctx, space, r, m * 32, "gl_poseidon_two_to_one_batch: r"));
    TRY(check_device_ptr(ctx, space, out, m * 32, "gl_poseidon_two_to_one_batch: out"));
    Guard g(ctx);
    const u64 *dl, *dr;
    TRY(stage_in(ctx, l, m * 32, space, 0, &dl));
    TRY(stage_in(ctx, r, m * 32, space, 1, &dr));
    u64* dout = out;
    if (space == GL_HOST) {
        void* t;
        TRY(scratch_get(ctx, 2, m * 32 + 8, &t));
        dout = (u64*)t;
    }
    launch_two_to_one_batch(dl, dr, dout, m, ctx->stream);
    TRY(copy_out(ctx, out, dout, m * 32, space));
    return finish(ctx);
}

extern "C" int gl_poseidon_hash_no_pad_batch(gl_ctx* ctx, const uint64_t* in, uint32_t len_each, uint64_t m,
                                             uint64_t* out, int space) {
    if (!ctx) return GL_E_ARG;
    if (m && (!out || (len_each && !in))) return fail(ctx, GL_E_ARG, "gl_poseidon_hash_no_pad_batch: NULL buffer");
    TRY(check_device_ptr(ctx, space, in, (size_t)m * len_each * 8, "gl_poseidon_hash_no_pad_batch: in"));
    TRY(check_device_ptr(ctx, space, out, m * 32, "gl_poseidon_hash_no_pad_batch: out"));
    Guard g(ctx);
    const u64* din;
    TRY(stage_in(ctx, in, (size_t)m * len_each * 8, space, 0, &din));
    u64* dout = out;
    if (space == GL_HOST) {
        void* t;
        TRY(scratch_get(ctx, 2, m * 32 + 8, &t));
        dout = (u64*)t;
    }
    launch_hash_no_pad_rows(din, len_each, m, dout, ctx->stream);
    TRY(copy_out(ctx, out, dout, m * 32, space));
    return finish(ctx);
}

extern "C" int gl_smt_leaf_hash_batch(gl_ctx* ctx, const uint64_t* keys, const uint64_t* values, uint64_t* out,
                                      uint64_t m, int space) {
    if (!ctx) return GL_E_ARG;
    if (m && (!keys || !values || !out)) return fail(ctx, GL_E_ARG, "gl_smt_leaf_hash_batch: NULL buffer");
    TRY(check_device_ptr(ctx, space, keys, m * 32, "gl_smt_leaf_hash_batch: keys"));
    TRY(check_device_ptr(ctx, space, values, m * 32, "gl_smt_leaf_hash_batch: values"));
    TRY(check_device_ptr(ctx, space, out, m * 32, "gl_smt_leaf_hash_batch: out"));
    Guard g(ctx);
    const u64 *dk, *dv;
    TRY(stage_in(ctx, keys, m * 32, space, 0, &dk));
    TRY(stage_in(ctx, values, m * 32, space, 1, &dv));
    u64* dout = out;
    if (space == GL_HOST) {
        void* t;
        TRY(scratch_get(ctx, 2, m * 32 + 8, &t));
        dout = (u64*)t;
    }
    launch_smt_leaf_hash_batch(dk, dv, dout, m, ctx->stream);
    TRY(copy_out(ctx, out, dout, m * 32, space));
    return finish(ctx);
}

extern "C" int gl_smt_verify_process_batch(gl_ctx* ctx, const gl_smt_proof_hdr* proofs, const uint64_t* sib_pool,
                                           const uint64_t* sib_off, uint64_t m, int32_t* status, int space) {
    if (!ctx) return GL_E_ARG;
    if (m == 0) return GL_OK;
    if (!proofs || !sib_off || !status) return fail(ctx, GL_E_ARG, "gl_smt_verify_process_batch: NULL buffer");
    TRY(check_device_ptr(ctx, space, proofs, m * sizeof(gl_smt_proof_hdr), "gl_smt_verify_process_batch: proofs"));
    // the pool's length is sib_off[m], which lies on the device: any non-empty pool holds 32-byte siblings
    TRY(check_device_ptr(ctx, space, sib_pool, 32, "gl_smt_verify_process_batch: sib_pool"));
    TRY(check_device_ptr(ctx, space, sib_off, (m + 1) * 8, "gl_smt_verify_process_batch: sib_off"));
    TRY(check_device_ptr(ctx, space, status, m * 4, "gl_smt_verify_process_batch: status"));
    Guard g(ctx);
    if (space == GL_DEVICE) {
        launch_smt_verify_process(proofs, sib_pool, sib_off, m, status, ctx->stream);
        return finish(ctx);
    }
    uint64_t total = sib_off[m];
    for (uint64_t t = 0; t < m; t++)
        if (sib_off[t + 1] < sib_off[t]) return fail(ctx, GL_E_ARG, "gl_smt_verify_process_batch: sib_off not monotone");
    if (total && !sib_pool) return fail(ctx, GL_E_ARG, "gl_smt_verify_process_batch: NULL sib_pool");
    const u64 *dp, *dpool, *doff;
    TRY(stage_in(ctx, proofs, m * sizeof(gl_smt_proof_hdr), GL_HOST, 0, &dp));
    TRY(stage_in(ctx, sib_pool, total * 32, GL_HOST, 1, &dpool));
    TRY(stage_in(ctx, sib_off, (m + 1) * 8, GL_HOST, 2, &doff));
    void* dst;
    TRY(scratch_get(ctx, 3, m * 4, &dst));
    launch_smt_verify_process((const gl_smt_proof_hdr*)dp, dpool, doff, m, (int*)dst, ctx->stream);
    TRY(copy_out(ctx, status, dst, m * 4, GL_HOST));
    return finish(ctx);
}

// ------------------------------------------------------------------------------------------------
// N2: bulk sparse Merkle tree
// ------------------------------------------------------------------------------------------------
extern "C" int gl_smt_build(gl_ctx* ctx, const uint64_t* keys, const uint64_t* values, uint64_t m, uint64_t* root_out,
                            uint64_t* nodes_out, uint64_t nodes_cap, uint64_t* num_nodes_out, uint64_t* leaf_hashes_out,
                            int space) {
    if (!ctx) return GL_E_ARG;
    if (!root_out || (m && (!keys || !values))) return fail(ctx, GL_E_ARG, "gl_smt_build: NULL buffer");
    if (m >= ((uint64_t)1 << 31)) return fail(ctx, GL_E_ARG, "gl_smt_build: at most 2^31 - 1 entries");
    TRY(check_device_ptr(ctx, space, keys, m * 32, "gl_smt_build: keys"));
    TRY(check_device_ptr(ctx, space, values, m * 32, "gl_smt_build: values"));
    TRY(check_device_ptr(ctx, space, root_out, 32, "gl_smt_build: root_out"));
    TRY(check_device_ptr(ctx, space, nodes_out, nodes_cap * 96, "gl_smt_build: nodes_out"));
    TRY(check_device_ptr(ctx, space, leaf_hashes_out, m * 32, "gl_smt_build: leaf_hashes_out"));
    Guard g(ctx);
    if (m == 0) {
        if (num_nodes_out) *num_nodes_out = 0;
        if (space == GL_HOST) memset(root_out, 0, 32);
        else CK(cudaMemsetAsync(root_out, 0, 32, ctx->stream));
        return finish(ctx);
    }
    smt_build_buffers b;
    memset(&b, 0, sizeof b);
    b.m = m;
    const u64 *dk, *dv;
    TRY(stage_in(ctx, keys, m * 32, space, 0, &dk));
    TRY(stage_in(ctx, values, m * 32, space, 1, &dv));
    b.keys = dk;
    b.values = dv;
    b.sort_tmp_bytes = smt_sort_temp_bytes(m);
    // one scratch block carved into the work arrays (all 8-byte aligned)
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t at = off; off += al(bytes); return at; };
    const size_t o_rk = take(m * 32), o_rka = take(m * 8), o_perm = take(m * 4), o_perma = take(m * 4), o_leafh = take(m * 32),
                 o_lcp = take(m * 2), o_vf = take(m * 32), o_vl = take(m * 32), o_end = take(m * 4), o_start = take(m * 4),
                 o_fd = take(m * 2), o_lv = take(m), o_hist = take(258 * 4), o_cnt = take(8), o_root = take(32),
                 o_tmp = take(b.sort_tmp_bytes), o_lh = take(leaf_hashes_out && space == GL_HOST ? m * 32 : 0),
                 o_nodes = take(nodes_out && space == GL_HOST ? nodes_cap * 96 : 0);
    void* base;
    TRY(scratch_get(ctx, 2, off, &base));
    char* p = (char*)base;
    b.rk = (u64*)(p + o_rk); b.rk_alt = (u64*)(p + o_rka); b.perm = (uint32_t*)(p + o_perm); b.perm_alt = (uint32_t*)(p + o_perma);
    b.leafh = (u64*)(p + o_leafh); b.lcp = (uint16_t*)(p + o_lcp); b.val_first = (u64*)(p + o_vf); b.val_last = (u64*)(p + o_vl);
    b.end_of = (uint32_t*)(p + o_end); b.start_of = (uint32_t*)(p + o_start); b.form_depth = (uint16_t*)(p + o_fd);
    b.last_valid = (uint8_t*)(p + o_lv); b.hist = (uint32_t*)(p + o_hist); b.node_count = (unsigned long long*)(p + o_cnt);
    b.sort_tmp = p + o_tmp;
    b.leaf_hashes = leaf_hashes_out ? (space == GL_HOST ? (u64*)(p + o_lh) : leaf_hashes_out) : nullptr;
    b.nodes = nodes_out ? (space == GL_HOST ? (u64*)(p + o_nodes) : nodes_out) : nullptr;
    b.nodes_cap = nodes_out ? nodes_cap : 0;
    u64* d_root = (u64*)(p + o_root);
    b.zero_values = b.hist + 257;
    CK(cudaMemsetAsync(b.hist, 0, 258 * 4, ctx->stream));
    CK(cudaMemsetAsync(b.node_count, 0, 8, ctx->stream));
    int rc = smt_build_prepare(b, ctx->stream);
    if (rc) return cuda_fail(ctx, (cudaError_t)rc, "gl_smt_build: sort");
    uint32_t hist[258];
    CK(cudaMemcpyAsync(hist, b.hist, sizeof hist, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (hist[257]) return fail(ctx, GL_E_ARG, "SparseMerkleTree::insert: value must be non-zero (src/smt/tree.rs: a zero value is a removal; use gl_smt_set_proofs for sequences with removals)");
    if (hist[256]) return fail(ctx, GL_E_ARG, "SparseMerkleTree::insert: given key already exists (duplicate keys in the batch)");
    int dmax = -1;
    for (int d = 255; d >= 0; d--)
        if (hist[d]) { dmax = d; break; }
    for (int d = dmax; d >= 0; d--) smt_build_level(b, (unsigned)d, ctx->stream);
    // m == 1: the single leaf is the root; else the group [0, m-1] climbed to depth 0
    CK(cudaMemcpyAsync(d_root, m == 1 ? b.leafh : b.val_first, 32, cudaMemcpyDeviceToDevice, ctx->stream));
    TRY(copy_out(ctx, root_out, d_root, 32, space));
    unsigned long long count = 0;
    CK(cudaMemcpyAsync(&count, b.node_count, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (num_nodes_out) *num_nodes_out = count;
    if (space == GL_HOST) {
        if (leaf_hashes_out) TRY(copy_out(ctx, leaf_hashes_out, b.leaf_hashes, m * 32, GL_HOST));
        if (nodes_out) TRY(copy_out(ctx, nodes_out, b.nodes, (count < nodes_cap ? count : nodes_cap) * 96, GL_HOST));
    }
    return finish(ctx);
}

// The sweep of smt_proofs.cu over m events already on the device: the first m_sets are `set` calls, the rest `find`
// queries.  Set mode (m_sets == m) writes m process proofs, find mode m - m_sets inclusion proofs.
static int smt_events_run(gl_ctx* ctx, const u64* dk, const u64* dv, uint64_t m, uint64_t m_sets, void* hdr_out,
                          uint64_t* sib_pool_out, uint64_t sib_cap, uint64_t* sib_off_out, uint64_t* num_siblings_out,
                          int space, const char* name) {
    const bool find_mode = m_sets < m;
    const uint64_t n_out = find_mode ? m - m_sets : m;
    smt_build_buffers b;
    memset(&b, 0, sizeof b);
    b.m = m;
    b.keys = dk;
    b.values = dv;
    b.sort_tmp_bytes = smt_sort_temp_bytes(m);
    const size_t tmp_bytes = std::max(b.sort_tmp_bytes, smt_proof_temp_bytes(m));
    const size_t hdr_bytes = find_mode ? n_out * sizeof(gl_smt_inclusion_hdr) : n_out * sizeof(gl_smt_proof_hdr);
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t at = off; off += al(bytes); return at; };
    const size_t o_rk = take(m * 32), o_rka = take(m * 8), o_perm = take(m * 4), o_perma = take(m * 4), o_leafh = take(m * 32),
                 o_lcp = take(m * 2), o_vf = take(m * 32), o_fd = take(m * 2), o_lv = take(m), o_hist = take(257 * 4 + 8),
                 o_tmp = take(tmp_bytes), o_u32 = take(19 * m * 4 + 64), o_val = take(2 * m * 32), o_keys = take(2 * m * 8),
                 o_off = take((m + 1) * 8), o_hdr = take(hdr_bytes);
    void* base;
    TRY(scratch_get(ctx, 2, off, &base));
    char* p0 = (char*)base;
    b.rk = (u64*)(p0 + o_rk); b.rk_alt = (u64*)(p0 + o_rka); b.perm = (uint32_t*)(p0 + o_perm); b.perm_alt = (uint32_t*)(p0 + o_perma);
    b.leafh = (u64*)(p0 + o_leafh); b.lcp = (uint16_t*)(p0 + o_lcp); b.val_first = (u64*)(p0 + o_vf);
    b.form_depth = (uint16_t*)(p0 + o_fd); b.last_valid = (uint8_t*)(p0 + o_lv); b.hist = (uint32_t*)(p0 + o_hist);
    b.sort_tmp = p0 + o_tmp;
    CK(cudaMemsetAsync(b.hist, 0, 257 * 4 + 8, ctx->stream));
    int rc = smt_build_prepare(b, ctx->stream);
    if (rc) return cuda_fail(ctx, (cudaError_t)rc, name);
    uint32_t hist[257];
    CK(cudaMemcpyAsync(hist, b.hist, sizeof hist, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    // hist[256] = adjacent events with the same key (updates, removals, re-inserts, queries)
    int dmax = -1;
    for (int d = 255; d >= 0; d--)
        if (hist[d]) { dmax = d; break; }
    smt_proof_buffers q;
    memset(&q, 0, sizeof q);
    q.m = m;
    q.m_sets = m_sets;
    q.bottom = (uint32_t)(dmax + 1);
    q.stride = q.bottom > 1 ? q.bottom : 1;
    q.keys = dk; q.values = dv; q.rk = b.rk; q.perm = b.perm; q.lcp = b.lcp; q.leafh = b.leafh;
    uint32_t* u = (uint32_t*)(p0 + o_u32);
    q.a_cur = u; q.end_cur = u + m; q.ord_cur = u + 2 * m; q.inv_cur = u + 3 * m; q.tm_cur = u + 4 * m;
    q.a_nxt = u + 5 * m; q.end_nxt = u + 6 * m; q.ord_nxt = u + 7 * m; q.inv_nxt = u + 8 * m; q.tm_nxt = u + 9 * m;
    q.stop_depth = u + 10 * m; q.stop_old = u + 11 * m;
    q.dc_cur = u + 12 * m; q.dc_nxt = u + 13 * m; q.rep_cur = u + 14 * m; q.rep_nxt = u + 15 * m; q.pos_of_time = u + 16 * m;
    q.deep_dc = u + 17 * m; q.deep_rep = u + 18 * m;
    q.val_cur = (u64*)(p0 + o_val); q.val_nxt = q.val_cur + 4 * m;
    if (find_mode) q.inc = (gl_smt_inclusion_hdr*)(p0 + o_hdr);
    else q.hdr = (gl_smt_proof_hdr*)(p0 + o_hdr);
    q.other = (uint32_t*)(p0 + o_keys);       // m * 4 bytes
    q.bit = (uint8_t*)(p0 + o_keys) + 4 * m;   // m bytes
    u64* d_off = (u64*)(p0 + o_off);
    // per-event sibling rows while sweeping: [m][stride][4]; counts (u32 [m + 1]) reuse the radix-sort double buffer
    PoolBuf d_sib;
    TRY(d_sib.alloc(ctx, (size_t)m * q.stride * 32));
    q.sib = d_sib.get();
    uint32_t* counts = (uint32_t*)b.rk_alt;   // m * 8 bytes >= (m + 1) * 4
    rc = smt_proofs_sweep(q, dmax, hist, counts, b.sort_tmp, tmp_bytes, ctx->stream);
    if (rc == 0) rc = smt_proofs_offsets(counts, d_off, m, b.sort_tmp, tmp_bytes, ctx->stream);
    if (rc) return cuda_fail(ctx, (cudaError_t)rc, name);
    u64 total = 0;
    cudaError_t e = cudaMemcpyAsync(&total, d_off + m, 8, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return cuda_fail(ctx, e, name);
    *num_siblings_out = total;
    PoolBuf d_pool;
    if (sib_pool_out && total <= sib_cap && total) {
        if (space == GL_DEVICE) {
            smt_proofs_gather(q, d_off, sib_cap, sib_pool_out, ctx->stream);
        } else {
            TRY(d_pool.alloc(ctx, (size_t)total * 32));
            smt_proofs_gather(q, d_off, total, d_pool.get(), ctx->stream);
            TRY(copy_out(ctx, sib_pool_out, d_pool.get(), d_pool.bytes(), GL_HOST));
        }
    }
    TRY(copy_out(ctx, hdr_out, p0 + o_hdr, hdr_bytes, space));
    // in find mode the sets have no siblings, so the offsets of the queries start at 0
    TRY(copy_out(ctx, sib_off_out, d_off + (m - n_out), (n_out + 1) * 8, space));
    return finish(ctx);
}

// N2, second half: the process proofs of m successive `set` calls on an empty tree (smt_proofs.cu)
extern "C" int gl_smt_set_proofs(gl_ctx* ctx, const uint64_t* keys, const uint64_t* values, uint64_t m,
                                 gl_smt_proof_hdr* proofs_out, uint64_t* sib_pool_out, uint64_t sib_cap,
                                 uint64_t* sib_off_out, uint64_t* num_siblings_out, int space) {
    if (!ctx) return GL_E_ARG;
    if (!num_siblings_out || (m && (!keys || !values || !proofs_out || !sib_off_out)))
        return fail(ctx, GL_E_ARG, "gl_smt_set_proofs: NULL buffer");
    if (m >= ((uint64_t)1 << 31)) return fail(ctx, GL_E_ARG, "gl_smt_set_proofs: at most 2^31 - 1 entries");
    *num_siblings_out = 0;
    if (m == 0) return GL_OK;
    TRY(check_device_ptr(ctx, space, keys, m * 32, "gl_smt_set_proofs: keys"));
    TRY(check_device_ptr(ctx, space, values, m * 32, "gl_smt_set_proofs: values"));
    TRY(check_device_ptr(ctx, space, proofs_out, m * sizeof(gl_smt_proof_hdr), "gl_smt_set_proofs: proofs_out"));
    TRY(check_device_ptr(ctx, space, sib_pool_out, sib_cap * 32, "gl_smt_set_proofs: sib_pool_out"));
    TRY(check_device_ptr(ctx, space, sib_off_out, (m + 1) * 8, "gl_smt_set_proofs: sib_off_out"));
    Guard g(ctx);
    const u64 *dk, *dv;
    TRY(stage_in(ctx, keys, m * 32, space, 0, &dk));
    TRY(stage_in(ctx, values, m * 32, space, 1, &dv));
    return smt_events_run(ctx, dk, dv, m, m, proofs_out, sib_pool_out, sib_cap, sib_off_out, num_siblings_out, space,
                          "gl_smt_set_proofs");
}

// tree.find for a batch of keys against the tree those sets leave
extern "C" int gl_smt_find_batch(gl_ctx* ctx, const uint64_t* keys, const uint64_t* values, uint64_t m, const uint64_t* queries,
                                 uint64_t nq, gl_smt_inclusion_hdr* proofs_out, uint64_t* sib_pool_out, uint64_t sib_cap,
                                 uint64_t* sib_off_out, uint64_t* num_siblings_out, int space) {
    if (!ctx) return GL_E_ARG;
    if (!num_siblings_out || (m && (!keys || !values)) || (nq && (!queries || !proofs_out || !sib_off_out)))
        return fail(ctx, GL_E_ARG, "gl_smt_find_batch: NULL buffer");
    if (m + nq >= ((uint64_t)1 << 31)) return fail(ctx, GL_E_ARG, "gl_smt_find_batch: at most 2^31 - 1 entries and queries");
    *num_siblings_out = 0;
    if (nq == 0) return GL_OK;
    TRY(check_device_ptr(ctx, space, keys, m * 32, "gl_smt_find_batch: keys"));
    TRY(check_device_ptr(ctx, space, values, m * 32, "gl_smt_find_batch: values"));
    TRY(check_device_ptr(ctx, space, queries, nq * 32, "gl_smt_find_batch: queries"));
    TRY(check_device_ptr(ctx, space, proofs_out, nq * sizeof(gl_smt_inclusion_hdr), "gl_smt_find_batch: proofs_out"));
    TRY(check_device_ptr(ctx, space, sib_pool_out, sib_cap * 32, "gl_smt_find_batch: sib_pool_out"));
    TRY(check_device_ptr(ctx, space, sib_off_out, (nq + 1) * 8, "gl_smt_find_batch: sib_off_out"));
    Guard g(ctx);
    // one event list on the device: the sets, then the queries (their values are not looked at)
    const uint64_t all = m + nq;
    void *k_all, *v_all;
    TRY(scratch_get(ctx, 0, all * 32, &k_all));
    TRY(scratch_get(ctx, 1, all * 32, &v_all));
    const cudaMemcpyKind kind = space == GL_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    if (m) {
        CK(cudaMemcpyAsync(k_all, keys, m * 32, kind, ctx->stream));
        CK(cudaMemcpyAsync(v_all, values, m * 32, kind, ctx->stream));
    }
    CK(cudaMemcpyAsync((char*)k_all + m * 32, queries, nq * 32, kind, ctx->stream));
    CK(cudaMemsetAsync((char*)v_all + m * 32, 0, nq * 32, ctx->stream));
    if (space == GL_HOST) CK(cudaStreamSynchronize(ctx->stream));   // the caller's arrays are free again
    return smt_events_run(ctx, (const u64*)k_all, (const u64*)v_all, all, m, proofs_out, sib_pool_out, sib_cap, sib_off_out,
                          num_siblings_out, space, "gl_smt_find_batch");
}

// verify_merkle_proof_to_cap for k (leaf, index, path) triples against one cap
extern "C" int gl_merkle_verify_batch(gl_ctx* ctx, const uint64_t* leaves, uint32_t leaf_len, const uint64_t* leaf_indices,
                                      const uint64_t* paths, uint32_t path_len, const uint64_t* cap, uint32_t cap_height,
                                      uint64_t k, int32_t* ok, int space) {
    if (!ctx) return GL_E_ARG;
    if (k && (!leaves || !leaf_indices || !cap || !ok || (path_len && !paths)))
        return fail(ctx, GL_E_ARG, "gl_merkle_verify_batch: NULL buffer");
    if (leaf_len == 0 || cap_height > 30 || path_len > 64) return fail(ctx, GL_E_ARG, "gl_merkle_verify_batch: bad shape");
    if (k == 0) return GL_OK;
    TRY(check_device_ptr(ctx, space, leaves, k * leaf_len * 8, "gl_merkle_verify_batch: leaves"));
    TRY(check_device_ptr(ctx, space, leaf_indices, k * 8, "gl_merkle_verify_batch: leaf_indices"));
    TRY(check_device_ptr(ctx, space, paths, k * (size_t)path_len * 32, "gl_merkle_verify_batch: paths"));
    TRY(check_device_ptr(ctx, space, cap, ((size_t)32) << cap_height, "gl_merkle_verify_batch: cap"));
    TRY(check_device_ptr(ctx, space, ok, k * 4, "gl_merkle_verify_batch: ok"));
    Guard g(ctx);
    const u64 *dl, *di, *dp, *dc;
    TRY(stage_in(ctx, leaves, k * leaf_len * 8, space, 0, &dl));
    TRY(stage_in(ctx, leaf_indices, k * 8, space, 1, &di));
    TRY(stage_in(ctx, paths, k * (size_t)path_len * 32, space, 2, &dp));
    TRY(stage_in(ctx, cap, ((size_t)32) << cap_height, space, 3, &dc));
    int* d_ok = (int*)ok;
    if (space == GL_HOST) {
        void* d;
        TRY(scratch_get(ctx, 4, k * 4, &d));
        d_ok = (int*)d;
    }
    launch_merkle_verify_batch(dl, leaf_len, di, dp, path_len, dc, cap_height, k, d_ok, ctx->stream);
    TRY(copy_out(ctx, ok, d_ok, k * 4, space));
    return finish(ctx);
}

// ------------------------------------------------------------------------------------------------
// MerkleTree::new on caller-provided row-major leaves
// ------------------------------------------------------------------------------------------------
extern "C" int gl_merkle_build(gl_ctx* ctx, const uint64_t* leaves, uint64_t num_leaves, uint32_t leaf_len,
                               uint32_t cap_height, uint64_t* digests_out, uint64_t* cap_out, int space) {
    if (!ctx) return GL_E_ARG;
    if (!is_pow2(num_leaves)) return fail(ctx, GL_E_ARG, "MerkleTree::new: number of leaves is not a power of two (log2_strict)");
    unsigned lg = ilog2(num_leaves);
    if (cap_height > lg)
        return fail(ctx, GL_E_ARG, "MerkleTree::new: cap_height must be at most log2(leaves.len())");
    if (!cap_out || (leaf_len && !leaves)) return fail(ctx, GL_E_ARG, "gl_merkle_build: NULL buffer");
    TRY(check_device_ptr(ctx, space, leaves, (size_t)num_leaves * leaf_len * 8, "gl_merkle_build: leaves"));
    TRY(check_device_ptr(ctx, space, digests_out, 2 * (num_leaves - ((uint64_t)1 << cap_height)) * 32, "gl_merkle_build: digests_out"));
    TRY(check_device_ptr(ctx, space, cap_out, ((size_t)32 << cap_height), "gl_merkle_build: cap_out"));
    Guard g(ctx);
    const u64* dl;
    TRY(stage_in(ctx, leaves, (size_t)num_leaves * leaf_len * 8, space, 0, &dl));
    uint64_t nd = 2 * (num_leaves - ((uint64_t)1 << cap_height));
    void *dd, *dc;
    TRY(scratch_get(ctx, 1, nd * 32 + 32, &dd));
    TRY(scratch_get(ctx, 2, ((size_t)32 << cap_height), &dc));
    launch_merkle_rows(dl, leaf_len, lg, cap_height, (u64*)dd, (u64*)dc, ctx->stream);
    TRY(copy_out(ctx, digests_out, dd, nd * 32, space));
    TRY(copy_out(ctx, cap_out, dc, ((size_t)32 << cap_height), space));
    return finish(ctx);
}

// ------------------------------------------------------------------------------------------------
// plonky2_field::fft batches
// ------------------------------------------------------------------------------------------------
static int fft_entry(gl_ctx* ctx, uint64_t* data, uint32_t log_n, uint32_t c, int space, bool inverse, bool coset,
                     uint64_t shift, const char* name) {
    if (!ctx) return GL_E_ARG;
    if (log_n > 30) return fail(ctx, GL_E_ARG, std::string(name) + ": log_n > 30 not supported");
    if (c == 0) return GL_OK;
    if (!data) return fail(ctx, GL_E_ARG, std::string(name) + ": NULL data");
    size_t bytes = ((size_t)c << log_n) * 8;
    TRY(check_device_ptr(ctx, space, data, bytes, (std::string(name) + ": data").c_str()));
    Guard g(ctx);
    const u64* d;
    TRY(stage_in(ctx, data, bytes, space, 0, &d));
    const u64 *pre = nullptr, *post = nullptr;
    if (coset) {
        u64 sh = glh::canon(shift);
        if (sh == 0) return fail(ctx, GL_E_ARG, std::string(name) + ": zero coset shift");
        if (!inverse) TRY(pow_table(ctx, sh, &pre));
        else TRY(pow_table(ctx, glh::inv(sh), &post));
    }
    TRY(transform_natural(ctx, (u64*)d, log_n, c, inverse, pre, post));
    TRY(copy_out(ctx, data, d, bytes, space));
    return finish(ctx);
}
extern "C" int gl_fft_batch(gl_ctx* ctx, uint64_t* data, uint32_t log_n, uint32_t c, int space) {
    return fft_entry(ctx, data, log_n, c, space, false, false, 1, "gl_fft_batch");
}
extern "C" int gl_ifft_batch(gl_ctx* ctx, uint64_t* data, uint32_t log_n, uint32_t c, int space) {
    return fft_entry(ctx, data, log_n, c, space, true, false, 1, "gl_ifft_batch");
}
extern "C" int gl_coset_fft_batch(gl_ctx* ctx, uint64_t* data, uint32_t log_n, uint32_t c, uint64_t shift, int space) {
    return fft_entry(ctx, data, log_n, c, space, false, true, shift, "gl_coset_fft_batch");
}
extern "C" int gl_coset_ifft_batch(gl_ctx* ctx, uint64_t* data, uint32_t log_n, uint32_t c, uint64_t shift, int space) {
    return fft_entry(ctx, data, log_n, c, space, true, true, shift, "gl_coset_ifft_batch");
}

// ------------------------------------------------------------------------------------------------
// PolynomialBatch::from_values / from_coeffs
// ------------------------------------------------------------------------------------------------
static void mark(gl_ctx* ctx, int i) { cudaEventRecord(ctx->ev[i], ctx->stream); }

// end of a successful commit: the streaming hash state goes back to the pool, the phase times are kept
static void commit_done(gl_ctx* ctx, gl_commit* h) {
    h->hstate.reset();
    for (int i = 0; i < GL_PHASES; i++) cudaEventElapsedTime(&ctx->phase_ms[i], ctx->ev[i], ctx->ev[i + 1]);
    ctx->ev_valid = true;
}

// A failed commit may still have copies in flight on the PCIe streams, which are not ordered with ctx->stream: every
// stream drains before the handle, and with it its blocks, is dropped.
static void quiesce(gl_ctx* ctx) {
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->h2d_stream);
    cudaStreamSynchronize(ctx->d2h_stream);
    cudaGetLastError();
}

static int commit_check(gl_ctx* ctx, uint32_t log_n, uint32_t c, uint32_t rate_bits, uint32_t cap_height,
                        const char* name) {
    if (c == 0) return fail(ctx, GL_E_ARG, std::string(name) + ": empty polynomial batch");
    if (log_n + rate_bits > 30) return fail(ctx, GL_E_ARG, std::string(name) + ": log_n + rate_bits > 30 not supported");
    if (cap_height > log_n + rate_bits)
        return fail(ctx, GL_E_ARG, std::string(name) + ": cap_height must be at most log2(leaves.len())");
    unsigned lc = ilog2(ctx->shard_count);
    if (lc > rate_bits || lc > cap_height)
        return fail(ctx, GL_E_ARG, std::string(name) + ": shard count must divide 2^rate_bits and 2^cap_height");
    return GL_OK;
}

// A polynomial commit of the ctx's shard with every block allocated: `coeff_cols` >= c coefficient columns, the LDE,
// the digests and the cap
static int commit_new(gl_ctx* ctx, uint32_t log_n, uint32_t c, uint32_t rate_bits, uint32_t cap_height, uint32_t salt,
                      uint32_t coeff_cols, std::unique_ptr<gl_commit>* out) {
    std::unique_ptr<gl_commit> h(new (std::nothrow) gl_commit());
    if (!h) return fail(ctx, GL_E_OOM, "host allocation failed");
    h->ctx = ctx; h->log_n = log_n; h->c = c; h->rate_bits = rate_bits; h->cap_height = cap_height; h->salt = salt;
    h->shard_index = ctx->shard_index; h->shard_count = ctx->shard_count;
    const unsigned lc = ilog2(h->shard_count);
    h->n_local = ((u64)1 << log_n) * ((1u << rate_bits) >> lc);
    h->leaf_begin = (u64)h->shard_index * h->n_local;
    h->cap_local_bits = cap_height - lc;
    h->num_digests = 2 * (h->n_local - ((u64)1 << h->cap_local_bits));
    TRY(h->coeffs.alloc(ctx, ((size_t)coeff_cols << log_n) * 8));
    TRY(h->lde.alloc(ctx, (size_t)leaf_len(h.get()) * h->n_local * 8));
    TRY(h->digests.alloc(ctx, h->num_digests * 32));
    TRY(h->cap.alloc(ctx, (size_t)32 << h->cap_local_bits));
    *out = std::move(h);
    return GL_OK;
}

// "FFT + blinding" for columns [col0, col0 + ncols): every local coset of those columns, written in leaf order
static int commit_lde_columns(gl_ctx* ctx, gl_commit* h, uint32_t col0, uint32_t ncols) {
    const u64 n = (u64)1 << h->log_n;
    const uint32_t blocks = (1u << h->rate_bits) >> ilog2(h->shard_count);
    const u64* pre;
    TRY(coset_tables(ctx, h->log_n, h->rate_bits, h->shard_index, h->shard_count, &pre));
    NttJob j;
    j.in = h->coeffs.get() + (size_t)col0 * n; j.in_ld = n; j.in_coset_stride = 0;
    j.out = h->lde.get() + (size_t)col0 * h->n_local; j.out_ld = h->n_local; j.out_coset_stride = n;
    j.L = h->log_n; j.columns = ncols; j.cosets = blocks; j.inverse = false; j.pre_tab = pre;
    j.pre_direct_ok = true;
    j.canonical_out = 1;
    return run_dif(ctx, j);
}

// "build Merkle tree"
static int commit_tree(gl_ctx* ctx, gl_commit* h, uint64_t* cap_out, int space, bool leaves_hashed = false) {
    const unsigned lg_local = h->log_n + h->rate_bits - ilog2(h->shard_count);
    if (h->salt) {
        // lde_values(): `.chain((0..salt_size).map(|_| F::rand_vec(degree << rate_bits)))` -- uniform field elements
        launch_salt_fill(h->lde.get() + (size_t)h->c * h->n_local, (u64)h->salt * h->n_local, ctx->salt_seed,
                         (ctx->salt_counter++ << 8) | h->shard_index, ctx->stream);
    }
    mark(ctx, 4);
    if (!leaves_hashed)
        launch_leaf_hash_cols(h->lde.get(), h->n_local, leaf_len(h), lg_local, h->cap_local_bits, h->digests.get(), h->cap.get(),
                              ctx->stream);
    mark(ctx, 5);
    launch_merkle_levels(lg_local, h->cap_local_bits, h->digests.get(), h->cap.get(), ctx->stream);
    mark(ctx, 6);
    if (cap_out) {
        uint64_t* dst = cap_out + 4 * ((size_t)h->shard_index << h->cap_local_bits);
        TRY(copy_out(ctx, dst, h->cap.get(), h->cap.bytes(), space));
    }
    return GL_OK;
}

// Streamed leaf hashing: polynomials [col0, col0 + ncols) have just been extended.  While the blocks come in polynomial
// order, every complete group of 8 polynomials (the sponge rate) is absorbed into the per-leaf Poseidon state right
// away, so the hashing overlaps the arrival of the next block; the last block closes the ragged group and writes the
// digests.  Out-of-order blocks switch the commit back to one hashing pass at the end.
static int commit_absorb_block(gl_ctx* ctx, gl_commit* h, uint32_t col0, uint32_t ncols) {
    if (!h->stream_hash) return GL_OK;
    if (col0 != h->next_col) {
        h->stream_hash = false;
        return GL_OK;
    }
    h->next_col += ncols;
    const uint32_t complete = h->next_col == h->c ? h->c : (h->next_col & ~7u);
    if (complete <= h->hashed_cols) return GL_OK;
    const bool first = h->hashed_cols == 0, last = complete == h->c;
    if (!h->hstate.get() && !(first && last)) TRY(h->hstate.alloc(ctx, (size_t)h->n_local * 12 * 8));
    const unsigned lg_local = h->log_n + h->rate_bits - ilog2(h->shard_count);
    launch_leaf_absorb_cols(h->lde.get(), h->n_local, h->hashed_cols, complete, lg_local, h->cap_local_bits, h->hstate.get(), first,
                            last, h->digests.get(), h->cap.get(), ctx->stream);
    h->hashed_cols = complete;
    return GL_OK;
}

// Where the polynomials of a host-side commit live: one [c][n] array, or one array per polynomial
// (Vec<PolynomialValues<F>> / Vec<PolynomialCoeffs<F>> as the reference holds them).
struct HostCols {
    uint64_t* flat = nullptr;
    uint64_t* const* cols = nullptr;
    explicit operator bool() const { return flat || cols; }
    void segs(uint32_t col0, uint32_t nc, u64 n, std::vector<staging::HostSeg>& out) const {
        out.clear();
        if (flat) {
            out.push_back({flat + (size_t)col0 * n, (size_t)nc * n * 8});
            return;
        }
        for (uint32_t j = 0; j < nc; j++) out.push_back({cols[col0 + j], (size_t)n * 8});
    }
};

// Host buffers: the H2D copy of column block b+1, the IFFT + LDE of block b and the D2H copy of block b's
// coefficients run on three streams, so PCIe traffic hides behind the transforms (PCIe is full duplex).
// Page-able arrays are packed into / unpacked from page-locked rings by helper threads (host_staging.h).
// polynomials per block of the host pipeline: about six blocks per commit, between 2 MB (launch overhead) and 96 MB
static uint32_t host_block_cols(const gl_commit* h) {
    const size_t col_bytes = ((size_t)1 << h->log_n) * 8;
    size_t block_bytes = (size_t)h->c * col_bytes / 6;
    if (block_bytes < ((size_t)2 << 20)) block_bytes = (size_t)2 << 20;
    if (block_bytes > ((size_t)96 << 20)) block_bytes = (size_t)96 << 20;
    uint32_t cb = (uint32_t)(block_bytes / col_bytes);
    if (cb < 1) cb = 1;
    if (cb > h->c) cb = h->c;
    return cb;
}
static uint32_t nblocks_host(const gl_commit* h) {
    const uint32_t cb = host_block_cols(h);
    return (h->c + cb - 1) / cb;
}

static int commit_pipeline_host(gl_ctx* ctx, gl_commit* h, const HostCols& input, bool is_values,
                                const HostCols& coeffs_out) {
    const u64 n = (u64)1 << h->log_n;
    const uint32_t cb = host_block_cols(h);
    // the first block is an eighth of the others: nothing runs under its upload, so it should be short
    const uint32_t cb0 = (cb >= 8 && h->c > cb) ? cb / 8 : cb;
    const uint32_t nb = 1 + (h->c - cb0 + cb - 1) / cb;
    while (ctx->pipe_ev.size() < 2 * (size_t)nb) {
        cudaEvent_t e;
        CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->pipe_ev.push_back(e);
    }
    cudaEvent_t start = ctx->ev[1];   // recorded by the caller on the main stream
    CK(cudaStreamWaitEvent(ctx->h2d_stream, start, 0));
    std::vector<staging::HostSeg> segs;
    uint32_t col0 = 0;
    for (uint32_t b = 0; col0 < h->c; b++) {
        const uint32_t want = b == 0 ? cb0 : cb;
        const uint32_t nc = (col0 + want <= h->c) ? want : h->c - col0;
        u64* dcol = h->coeffs.get() + (size_t)col0 * n;
        input.segs(col0, nc, n, segs);
        TRY(h2d_copy(ctx, dcol, segs.data(), segs.size(), ctx->h2d_stream));
        CK(cudaEventRecord(ctx->pipe_ev[2 * b], ctx->h2d_stream));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->pipe_ev[2 * b], 0));
        if (is_values) {
            TRY(transform_natural(ctx, dcol, h->log_n, nc, true, nullptr, nullptr));  // "IFFT"
            if (coeffs_out) {
                CK(cudaEventRecord(ctx->pipe_ev[2 * b + 1], ctx->stream));
                coeffs_out.segs(col0, nc, n, segs);
                TRY(d2h_copy(ctx, segs, dcol, ctx->pipe_ev[2 * b + 1]));
            }
        }
        TRY(commit_lde_columns(ctx, h, col0, nc));
        TRY(commit_absorb_block(ctx, h, col0, nc));   // hashing of what has arrived runs under the next block's PCIe time
        col0 += nc;
    }
    return GL_OK;
}

// copy-in, IFFT, LDE and tree of the freshly allocated commit `h`
static int commit_build(gl_ctx* ctx, gl_commit* h, const HostCols& input, bool is_values, const HostCols& coeffs_out,
                        uint64_t* cap_out, int space) {
    mark(ctx, 0);
    if (space == GL_HOST) {
        // phases 1..3 overlap in this mode: their sum is reported as "lde_ntt" (phase 3)
        mark(ctx, 1);
        mark(ctx, 2);
        mark(ctx, 3);
        h->stream_hash = h->c > 4 && nblocks_host(h) > 1 && !h->salt;   // the salt columns only exist at the end
        TRY(commit_pipeline_host(ctx, h, input, is_values, coeffs_out));
    } else {
        if (!is_values) {
            cudaError_t e = cudaMemcpyAsync(h->coeffs.get(), input.flat, h->coeffs.bytes(), cudaMemcpyDeviceToDevice, ctx->stream);
            if (e != cudaSuccess) return cuda_fail(ctx, e, "copy polynomials");
        }
        mark(ctx, 1);
        if (is_values) {
            // "IFFT": reads the caller's values where they lie, the coefficients land behind the handle
            TRY(transform_natural(ctx, h->coeffs.get(), h->log_n, h->c, true, nullptr, nullptr, input.flat));
            mark(ctx, 2);
            TRY(copy_out(ctx, coeffs_out.flat, h->coeffs.get(), h->coeffs.bytes(), space));
        } else {
            mark(ctx, 2);
        }
        mark(ctx, 3);
        TRY(commit_lde_columns(ctx, h, 0, h->c));
    }
    TRY(commit_tree(ctx, h, cap_out, space, h->stream_hash && h->hashed_cols == h->c));
    return finish(ctx);
}

// A whole polynomial commit with the ctx held (Guard): checks, allocation, build.  *out is set only on success.
static int commit_make(gl_ctx* ctx, const HostCols& input, bool is_values, uint32_t log_n, uint32_t c, uint32_t rate_bits,
                       uint32_t cap_height, const HostCols& coeffs_out, uint64_t* cap_out, int space, const char* name,
                       bool blinding, std::unique_ptr<gl_commit>* out) {
    TRY(commit_check(ctx, log_n, c, rate_bits, cap_height, name));
    if (input.cols || coeffs_out.cols) {
        for (uint32_t j = 0; j < c; j++)
            if ((input.cols && !input.cols[j]) || (coeffs_out.cols && !coeffs_out.cols[j]))
                return fail(ctx, GL_E_ARG, std::string(name) + ": NULL polynomial pointer");
    }
    std::unique_ptr<gl_commit> h;
    int rc = commit_new(ctx, log_n, c, rate_bits, cap_height, blinding ? GL_SALT_SIZE : 0, c, &h);
    if (rc == GL_OK) rc = commit_build(ctx, h.get(), input, is_values, coeffs_out, cap_out, space);
    if (space == GL_HOST) {   // coefficient downloads (also after an error: they write into caller memory)
        int rc2 = downloads_wait(ctx);
        if (rc == GL_OK) rc = rc2;
    }
    if (rc != GL_OK) {
        quiesce(ctx);
        return rc;
    }
    commit_done(ctx, h.get());
    *out = std::move(h);
    return GL_OK;
}

static int commit_common(gl_ctx* ctx, const HostCols& input, bool is_values, uint32_t log_n, uint32_t c,
                         uint32_t rate_bits, uint32_t cap_height, const HostCols& coeffs_out, uint64_t* cap_out,
                         gl_commit** handle, int space, const char* name, bool blinding = false) {
    if (!ctx) return GL_E_ARG;
    if (!handle || !input) return fail(ctx, GL_E_ARG, std::string(name) + ": NULL argument");
    *handle = nullptr;
    TRY(commit_check(ctx, log_n, c, rate_bits, cap_height, name));   // the buffer sizes below need a valid geometry
    const size_t bytes = ((size_t)c << log_n) * 8;
    const std::string nm(name);
    TRY(check_device_ptr(ctx, space, input.flat, bytes, (nm + (is_values ? ": values" : ": coeffs")).c_str()));
    TRY(check_device_ptr(ctx, space, coeffs_out.flat, bytes, (nm + ": coeffs_out").c_str()));
    TRY(check_device_ptr(ctx, space, cap_out, (size_t)32 << cap_height, (nm + ": cap_out").c_str()));
    Guard g(ctx);
    std::unique_ptr<gl_commit> h;
    TRY(commit_make(ctx, input, is_values, log_n, c, rate_bits, cap_height, coeffs_out, cap_out, space, name, blinding, &h));
    *handle = h.release();
    return GL_OK;
}

extern "C" int gl_commit_from_values(gl_ctx* ctx, const uint64_t* values, uint32_t log_n, uint32_t c,
                                     uint32_t rate_bits, uint32_t cap_height, uint64_t* coeffs_out, uint64_t* cap_out,
                                     gl_commit** handle, int space) {
    HostCols in, out;
    in.flat = const_cast<uint64_t*>(values);
    out.flat = coeffs_out;
    return commit_common(ctx, in, true, log_n, c, rate_bits, cap_height, out, cap_out, handle, space,
                         "PolynomialBatch::from_values");
}
extern "C" int gl_commit_from_coeffs(gl_ctx* ctx, const uint64_t* coeffs, uint32_t log_n, uint32_t c,
                                     uint32_t rate_bits, uint32_t cap_height, uint64_t* cap_out, gl_commit** handle,
                                     int space) {
    HostCols in;
    in.flat = const_cast<uint64_t*>(coeffs);
    return commit_common(ctx, in, false, log_n, c, rate_bits, cap_height, HostCols(), cap_out, handle, space,
                         "PolynomialBatch::from_coeffs");
}
// One host array per polynomial, as the reference holds them (Vec<PolynomialValues<F>>, Vec<PolynomialCoeffs<F>>).
extern "C" int gl_commit_from_values_cols(gl_ctx* ctx, const uint64_t* const* values, uint32_t log_n, uint32_t c,
                                          uint32_t rate_bits, uint32_t cap_height, uint64_t* const* coeffs_out,
                                          uint64_t* cap_out, gl_commit** handle) {
    HostCols in, out;
    in.cols = const_cast<uint64_t* const*>(values);
    out.cols = coeffs_out;
    return commit_common(ctx, in, true, log_n, c, rate_bits, cap_height, out, cap_out, handle, GL_HOST,
                         "PolynomialBatch::from_values");
}
extern "C" int gl_commit_from_coeffs_cols(gl_ctx* ctx, const uint64_t* const* coeffs, uint32_t log_n, uint32_t c,
                                          uint32_t rate_bits, uint32_t cap_height, uint64_t* cap_out,
                                          gl_commit** handle) {
    HostCols in;
    in.cols = const_cast<uint64_t* const*>(coeffs);
    return commit_common(ctx, in, false, log_n, c, rate_bits, cap_height, HostCols(), cap_out, handle, GL_HOST,
                         "PolynomialBatch::from_coeffs");
}

// upstream's full signatures: from_values(values, rate_bits, blinding, cap_height, ..) / from_coeffs(..)
extern "C" int gl_commit_from_values_ex(gl_ctx* ctx, const uint64_t* values, const uint64_t* const* values_cols, uint32_t log_n,
                                        uint32_t c, uint32_t rate_bits, uint32_t blinding, uint32_t cap_height,
                                        uint64_t* coeffs_out, uint64_t* const* coeffs_out_cols, uint64_t* cap_out,
                                        gl_commit** handle, int space) {
    if (!ctx) return GL_E_ARG;
    if ((values != nullptr) == (values_cols != nullptr))
        return fail(ctx, GL_E_ARG, "PolynomialBatch::from_values: pass the polynomials either as one array or as one array each");
    if (values_cols && space != GL_HOST) return fail(ctx, GL_E_ARG, "PolynomialBatch::from_values: per-polynomial arrays are host memory");
    HostCols in, out;
    in.flat = const_cast<uint64_t*>(values);
    in.cols = const_cast<uint64_t* const*>(values_cols);
    if (values_cols) out.cols = coeffs_out_cols;
    else out.flat = coeffs_out;
    return commit_common(ctx, in, true, log_n, c, rate_bits, cap_height, out, cap_out, handle, space,
                         "PolynomialBatch::from_values", blinding != 0);
}
extern "C" int gl_commit_from_coeffs_ex(gl_ctx* ctx, const uint64_t* coeffs, const uint64_t* const* coeffs_cols, uint32_t log_n,
                                        uint32_t c, uint32_t rate_bits, uint32_t blinding, uint32_t cap_height, uint64_t* cap_out,
                                        gl_commit** handle, int space) {
    if (!ctx) return GL_E_ARG;
    if ((coeffs != nullptr) == (coeffs_cols != nullptr))
        return fail(ctx, GL_E_ARG, "PolynomialBatch::from_coeffs: pass the polynomials either as one array or as one array each");
    if (coeffs_cols && space != GL_HOST) return fail(ctx, GL_E_ARG, "PolynomialBatch::from_coeffs: per-polynomial arrays are host memory");
    HostCols in;
    in.flat = const_cast<uint64_t*>(coeffs);
    in.cols = const_cast<uint64_t* const*>(coeffs_cols);
    return commit_common(ctx, in, false, log_n, c, rate_bits, cap_height, HostCols(), cap_out, handle, space,
                         "PolynomialBatch::from_coeffs", blinding != 0);
}
extern "C" int gl_ctx_set_salt_seed(gl_ctx* ctx, uint64_t seed) {
    if (!ctx) return GL_E_ARG;
    Guard g(ctx);
    ctx->salt_seed = seed;
    ctx->salt_counter = 0;
    return GL_OK;
}
extern "C" int gl_commit_leaf_len(const gl_commit* h, uint32_t* len) {
    if (!h || !len) return GL_E_ARG;
    *len = leaf_len(h);
    return GL_OK;
}

extern "C" int gl_commit_begin(gl_ctx* ctx, uint32_t log_n, uint32_t c, uint32_t rate_bits, uint32_t cap_height,
                               gl_commit** handle) {
    return gl_commit_begin_ex(ctx, log_n, c, rate_bits, cap_height, 0, handle);
}
extern "C" int gl_commit_begin_ex(gl_ctx* ctx, uint32_t log_n, uint32_t c, uint32_t rate_bits, uint32_t cap_height,
                                  uint32_t flags, gl_commit** handle) {
    if (!ctx) return GL_E_ARG;
    if (!handle) return fail(ctx, GL_E_ARG, "gl_commit_begin: NULL handle");
    if (flags & ~(uint32_t)(GL_COMMIT_STREAM_HASH | GL_COMMIT_BLINDING)) return fail(ctx, GL_E_ARG, "gl_commit_begin_ex: unknown flag");
    *handle = nullptr;
    TRY(commit_check(ctx, log_n, c, rate_bits, cap_height, "PolynomialBatch::from_coeffs"));
    Guard g(ctx);
    std::unique_ptr<gl_commit> h;
    TRY(commit_new(ctx, log_n, c, rate_bits, cap_height, (flags & GL_COMMIT_BLINDING) ? GL_SALT_SIZE : 0, c, &h));
    h->finished = false;
    // <= 4 polynomials: hash_or_noop copies, nothing to absorb; salted leaves: the salt columns only exist at the end
    h->stream_hash = (flags & GL_COMMIT_STREAM_HASH) && c > 4 && !h->salt;
    for (int i = 0; i <= 3; i++) mark(ctx, i);
    *handle = h.release();
    return GL_OK;
}
extern "C" int gl_commit_add_coeffs(gl_commit* h, uint32_t col0, uint32_t ncols, const uint64_t* coeffs, int space) {
    if (!h) return GL_E_ARG;
    gl_ctx* ctx = h->ctx;
    if (h->finished) return fail(ctx, GL_E_STATE, "gl_commit_add_coeffs: the commit is already finished");
    if (!coeffs || ncols == 0 || col0 + (uint64_t)ncols > h->c) return fail(ctx, GL_E_ARG, "gl_commit_add_coeffs: bad column range");
    const u64 n = (u64)1 << h->log_n;
    TRY(check_device_ptr(ctx, space, coeffs, (size_t)ncols * n * 8, "gl_commit_add_coeffs: coeffs"));
    Guard g(ctx);
    CK(cudaMemcpyAsync(h->coeffs.get() + (size_t)col0 * n, coeffs, (size_t)ncols * n * 8,
                       space == GL_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));
    TRY(commit_lde_columns(ctx, h, col0, ncols));
    h->cols_added += ncols;
    TRY(commit_absorb_block(ctx, h, col0, ncols));
    return finish(ctx);
}
extern "C" int gl_commit_finish(gl_commit* h, uint64_t* cap_out, int space) {
    if (!h) return GL_E_ARG;
    gl_ctx* ctx = h->ctx;
    if (h->finished) return fail(ctx, GL_E_STATE, "gl_commit_finish: the commit is already finished");
    if (h->cols_added != h->c) return fail(ctx, GL_E_STATE, "gl_commit_finish: not every polynomial has been added");
    TRY(check_device_ptr(ctx, space, cap_out, (size_t)32 << h->cap_height, "gl_commit_finish: cap_out"));
    Guard g(ctx);
    TRY(commit_tree(ctx, h, cap_out, space, h->stream_hash && h->hashed_cols == h->c));
    TRY(finish(ctx));
    h->finished = true;
    commit_done(ctx, h);
    return GL_OK;
}

extern "C" void gl_commit_free(gl_commit* h) {
    if (!h) return;
    gl_ctx* ctx = h->ctx;
    Guard g(ctx);
    cudaStreamSynchronize(ctx->stream);
    delete h;
}

extern "C" int gl_commit_info(const gl_commit* h, uint32_t* log_n, uint32_t* c, uint32_t* rate_bits,
                              uint32_t* cap_height, uint64_t* leaf_begin, uint64_t* leaf_end) {
    if (!h) return GL_E_ARG;
    if (log_n) *log_n = h->log_n;
    if (c) *c = h->c;
    if (rate_bits) *rate_bits = h->rate_bits;
    if (cap_height) *cap_height = h->cap_height;
    if (leaf_begin) *leaf_begin = h->leaf_begin;
    if (leaf_end) *leaf_end = h->leaf_begin + h->n_local;
    return GL_OK;
}

extern "C" int gl_commit_device_ptrs(const gl_commit* h, const uint64_t** lde_cols, uint64_t* ld,
                                     const uint64_t** digests) {
    if (!h) return GL_E_ARG;
    if (lde_cols) *lde_cols = h->lde.get();
    if (ld) *ld = h->n_local;
    if (digests) *digests = h->digests.get();
    return GL_OK;
}

extern "C" int gl_commit_coeffs(gl_commit* h, uint64_t* coeffs_out, int space) {
    if (!h || !coeffs_out) return GL_E_ARG;
    gl_ctx* ctx = h->ctx;
    if (!h->coeffs.get()) return fail(ctx, GL_E_STATE, "gl_commit_coeffs: this handle has no polynomials (FRI layer tree)");
    TRY(check_device_ptr(ctx, space, coeffs_out, ((size_t)h->c << h->log_n) * 8, "gl_commit_coeffs: coeffs_out"));
    Guard g(ctx);
    TRY(copy_out(ctx, coeffs_out, h->coeffs.get(), ((size_t)h->c << h->log_n) * 8, space));
    return finish(ctx);
}

// Polynomials [col0, col0 + ncols) of the commit at one extension point -> values_out [ncols][2], with the ctx held
static int commit_eval(gl_ctx* ctx, const gl_commit* h, uint32_t col0, uint32_t ncols, const uint64_t point[2],
                       uint64_t* values_out, int space) {
    const u64 n = (u64)1 << h->log_n;
    const u64 chunks = (n + FRI_EVAL_CHUNK - 1) / FRI_EVAL_CHUNK;
    const glh::ext z = {glh::canon(point[0]), glh::canon(point[1])};
    const glh::ext z256 = glh::ext_pow(z, 256), zc = glh::ext_pow(z, FRI_EVAL_CHUNK);
    const u64 zz[2] = {z.a, z.b}, z2[2] = {z256.a, z256.b}, z3[2] = {zc.a, zc.b};
    void* d;
    TRY(scratch_get(ctx, 0, ((size_t)ncols * chunks + ncols) * 16, &d));
    u64* partial = (u64*)d;
    u64* d_out = space == GL_DEVICE ? values_out : partial + 2 * (size_t)ncols * chunks;
    launch_eval_at(h->coeffs.get() + (size_t)col0 * n, n, ncols, zz, z2, z3, partial, d_out, ctx->stream);
    if (space == GL_HOST) TRY(copy_out(ctx, values_out, d_out, (size_t)ncols * 16, GL_HOST));
    return GL_OK;
}

// OpeningSet::new: every polynomial of the commit at one extension point, without bringing the coefficients back
extern "C" int gl_commit_eval(gl_commit* h, const uint64_t point[2], uint64_t* values_out, int space) {
    if (!h || !point || !values_out) return GL_E_ARG;
    gl_ctx* ctx = h->ctx;
    if (!h->coeffs.get()) return fail(ctx, GL_E_STATE, "gl_commit_eval: this handle has no polynomials (FRI layer tree)");
    if (!h->finished && h->cols_added != h->c) return fail(ctx, GL_E_STATE, "gl_commit_eval: not every polynomial has been added");
    TRY(check_device_ptr(ctx, space, values_out, (size_t)h->c * 16, "gl_commit_eval: values_out"));
    Guard g(ctx);
    TRY(commit_eval(ctx, h, 0, h->c, point, values_out, space));
    return finish(ctx);
}

extern "C" int gl_commit_download(gl_commit* h, uint64_t* leaves_out, uint64_t* digests_out, int space) {
    if (!h) return GL_E_ARG;
    gl_ctx* ctx = h->ctx;
    if (!h->finished) return fail(ctx, GL_E_STATE, "gl_commit_download: gl_commit_finish has not run yet");
    TRY(check_device_ptr(ctx, space, leaves_out, (size_t)h->n_local * leaf_len(h) * 8, "gl_commit_download: leaves_out"));
    TRY(check_device_ptr(ctx, space, digests_out, h->num_digests * 32, "gl_commit_download: digests_out"));
    Guard g(ctx);
    if (digests_out) TRY(copy_out(ctx, digests_out, h->digests.get(), h->num_digests * 32, space));
    if (leaves_out) {
        if (space == GL_DEVICE) {
            launch_transpose_to_rows(h->lde.get(), h->n_local, leaf_len(h), 0, h->n_local, leaves_out, ctx->stream);
        } else {
            const u64 chunk = h->n_local < ((u64)1 << 16) ? h->n_local : ((u64)1 << 16);
            void* stage;
            TRY(scratch_get(ctx, 0, (size_t)chunk * leaf_len(h) * 8, &stage));
            for (u64 r0 = 0; r0 < h->n_local; r0 += chunk) {
                launch_transpose_to_rows(h->lde.get(), h->n_local, leaf_len(h), r0, chunk, (u64*)stage, ctx->stream);
                TRY(copy_out(ctx, leaves_out + (size_t)r0 * leaf_len(h), stage, (size_t)chunk * leaf_len(h) * 8, GL_HOST));
                CK(cudaStreamSynchronize(ctx->stream));   // `stage` is reused by the next chunk
            }
        }
    }
    return finish(ctx);
}

// local leaf indices on the device in scratch slot 3
static int upload_indices(gl_ctx* ctx, const gl_commit* h, const std::vector<u64>& local, const u64** d_idx) {
    (void)h;
    void* d;
    TRY(scratch_get(ctx, 3, local.size() * 8 + 8, &d));
    CK(cudaMemcpyAsync(d, local.data(), local.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    *d_idx = (const u64*)d;
    return GL_OK;
}

static int fetch_indices(gl_ctx* ctx, const uint64_t* idx, uint32_t k, int space, std::vector<u64>& host) {
    host.resize(k);
    if (space == GL_DEVICE) {
        CK(cudaMemcpyAsync(host.data(), idx, (size_t)k * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    } else {
        memcpy(host.data(), idx, (size_t)k * 8);
    }
    return GL_OK;
}

extern "C" int gl_commit_open(gl_commit* h, const uint64_t* leaf_indices, uint32_t k, uint64_t* rows_out,
                              uint64_t* paths_out, int space) {
    if (!h) return GL_E_ARG;
    gl_ctx* ctx = h->ctx;
    if (!h->finished) return fail(ctx, GL_E_STATE, "gl_commit_open: gl_commit_finish has not run yet");
    if (k == 0) return GL_OK;
    if (!leaf_indices) return fail(ctx, GL_E_ARG, "gl_commit_open: NULL indices");
    const unsigned sub_bits = h->log_n + h->rate_bits - h->cap_height;
    TRY(check_device_ptr(ctx, space, leaf_indices, (size_t)k * 8, "gl_commit_open: leaf_indices"));
    TRY(check_device_ptr(ctx, space, rows_out, (size_t)k * leaf_len(h) * 8, "gl_commit_open: rows_out"));
    TRY(check_device_ptr(ctx, space, paths_out, (size_t)k * sub_bits * 32, "gl_commit_open: paths_out"));
    Guard g(ctx);
    std::vector<u64> idx;
    TRY(fetch_indices(ctx, leaf_indices, k, space, idx));
    for (auto& v : idx) {
        if (v < h->leaf_begin || v >= h->leaf_begin + h->n_local)
            return fail(ctx, GL_E_ARG, "MerkleTree::get / prove: leaf index out of range for this shard");
        v -= h->leaf_begin;
    }
    const u64* d_idx;
    TRY(upload_indices(ctx, h, idx, &d_idx));
    if (rows_out) {
        u64* d_rows = rows_out;
        if (space == GL_HOST) {
            void* t;
            TRY(scratch_get(ctx, 0, (size_t)k * leaf_len(h) * 8, &t));
            d_rows = (u64*)t;
        }
        launch_gather_rows(h->lde.get(), h->n_local, leaf_len(h), d_idx, k, d_rows, ctx->stream);
        TRY(copy_out(ctx, rows_out, d_rows, (size_t)k * leaf_len(h) * 8, space));
    }
    if (paths_out && sub_bits) {
        u64* d_paths = paths_out;
        if (space == GL_HOST) {
            void* t;
            TRY(scratch_get(ctx, 1, (size_t)k * sub_bits * 32, &t));
            d_paths = (u64*)t;
        }
        launch_gather_paths(h->digests.get(), sub_bits, d_idx, k, d_paths, ctx->stream);
        TRY(copy_out(ctx, paths_out, d_paths, (size_t)k * sub_bits * 32, space));
    }
    return finish(ctx);
}

extern "C" int gl_commit_get_lde_values(gl_commit* h, const uint64_t* indices, uint32_t k, uint64_t step,
                                        uint64_t* rows_out, int space) {
    if (!h) return GL_E_ARG;
    gl_ctx* ctx = h->ctx;
    if (!h->finished) return fail(ctx, GL_E_STATE, "gl_commit_get_lde_values: gl_commit_finish has not run yet");
    if (k == 0) return GL_OK;
    if (!indices || !rows_out) return fail(ctx, GL_E_ARG, "gl_commit_get_lde_values: NULL buffer");
    TRY(check_device_ptr(ctx, space, indices, (size_t)k * 8, "gl_commit_get_lde_values: indices"));
    TRY(check_device_ptr(ctx, space, rows_out, (size_t)k * h->c * 8, "gl_commit_get_lde_values: rows_out"));
    Guard g(ctx);
    std::vector<u64> idx;
    TRY(fetch_indices(ctx, indices, k, space, idx));
    const unsigned lgN = h->log_n + h->rate_bits;
    for (auto& v : idx) {
        unsigned __int128 prod = (unsigned __int128)v * step;
        if (prod >= ((unsigned __int128)1 << lgN)) return fail(ctx, GL_E_ARG, "get_lde_values: index * step out of range");
        u64 leaf = bitrev((u64)prod, lgN);
        if (leaf < h->leaf_begin || leaf >= h->leaf_begin + h->n_local)
            return fail(ctx, GL_E_ARG, "get_lde_values: row not held by this shard");
        v = leaf - h->leaf_begin;
    }
    const u64* d_idx;
    TRY(upload_indices(ctx, h, idx, &d_idx));
    u64* d_rows = rows_out;
    if (space == GL_HOST) {
        void* t;
        TRY(scratch_get(ctx, 0, (size_t)k * h->c * 8, &t));
        d_rows = (u64*)t;
    }
    launch_gather_rows(h->lde.get(), h->n_local, h->c, d_idx, k, d_rows, ctx->stream);
    TRY(copy_out(ctx, rows_out, d_rows, (size_t)k * h->c * 8, space));
    return finish(ctx);
}

// ------------------------------------------------------------------------------------------------
// FRI layer commit / fold / proof of work
// ------------------------------------------------------------------------------------------------
extern "C" int gl_fri_layer_tree(gl_ctx* ctx, const uint64_t* values_ext, uint64_t len, uint32_t arity_bits,
                                 uint32_t cap_height, uint64_t* digests_out, uint64_t* cap_out, int space) {
    if (!ctx) return GL_E_ARG;
    if (!is_pow2(len)) return fail(ctx, GL_E_ARG, "fri_committed_trees: length is not a power of two");
    unsigned lg = ilog2(len);
    if (arity_bits > lg) return fail(ctx, GL_E_ARG, "fri_committed_trees: arity larger than the layer");
    if (cap_height > lg - arity_bits)
        return fail(ctx, GL_E_ARG, "MerkleTree::new: cap_height must be at most log2(leaves.len())");
    if (!values_ext || !cap_out) return fail(ctx, GL_E_ARG, "gl_fri_layer_tree: NULL buffer");
    TRY(check_device_ptr(ctx, space, values_ext, len * 16, "gl_fri_layer_tree: values_ext"));
    TRY(check_device_ptr(ctx, space, digests_out, 2 * ((len >> arity_bits) - ((uint64_t)1 << cap_height)) * 32,
                         "gl_fri_layer_tree: digests_out"));
    TRY(check_device_ptr(ctx, space, cap_out, (size_t)32 << cap_height, "gl_fri_layer_tree: cap_out"));
    Guard g(ctx);
    const u64* dv;
    TRY(stage_in(ctx, values_ext, len * 16, space, 0, &dv));
    const u64 nl = len >> arity_bits;
    const uint32_t cols = 2u << arity_bits;
    void *dcols, *dd, *dc;
    TRY(scratch_get(ctx, 1, len * 16, &dcols));
    uint64_t nd = 2 * (nl - ((uint64_t)1 << cap_height));
    TRY(scratch_get(ctx, 2, nd * 32 + 32, &dd));
    TRY(scratch_get(ctx, 3, (size_t)32 << cap_height, &dc));
    launch_fri_leaves(dv, lg, arity_bits, (u64*)dcols, ctx->stream);
    launch_merkle_cols((const u64*)dcols, nl, cols, lg - arity_bits, cap_height, (u64*)dd, (u64*)dc, ctx->stream);
    TRY(copy_out(ctx, digests_out, dd, nd * 32, space));
    TRY(copy_out(ctx, cap_out, dc, (size_t)32 << cap_height, space));
    return finish(ctx);
}

// A FRI layer tree kept on the device: the leaves are the arity-sized cosets of `values` ([2^lg][2] extension
// elements on the device), 2 << arity_bits columns each, with no polynomials behind the handle
static int fri_tree_new(gl_ctx* ctx, const u64* values, unsigned lg, unsigned arity_bits, uint32_t cap_height,
                        std::unique_ptr<gl_commit>* out) {
    std::unique_ptr<gl_commit> t(new (std::nothrow) gl_commit());
    if (!t) return fail(ctx, GL_E_OOM, "host allocation failed");
    t->ctx = ctx; t->log_n = lg - arity_bits; t->c = 2u << arity_bits; t->rate_bits = 0; t->cap_height = cap_height;
    t->n_local = (u64)1 << t->log_n; t->cap_local_bits = cap_height;
    t->num_digests = 2 * (t->n_local - ((u64)1 << cap_height));
    TRY(t->lde.alloc(ctx, (size_t)16 << lg));
    TRY(t->digests.alloc(ctx, t->num_digests * 32));
    TRY(t->cap.alloc(ctx, (size_t)32 << cap_height));
    launch_fri_leaves(values, lg, arity_bits, t->lde.get(), ctx->stream);
    launch_merkle_cols(t->lde.get(), t->n_local, t->c, t->log_n, cap_height, t->digests.get(), t->cap.get(), ctx->stream);
    *out = std::move(t);
    return GL_OK;
}

extern "C" int gl_fri_layer_commit(gl_ctx* ctx, const uint64_t* values_ext, uint64_t len, uint32_t arity_bits,
                                   uint32_t cap_height, uint64_t* cap_out, gl_commit** handle, int space) {
    if (!ctx) return GL_E_ARG;
    if (!handle) return fail(ctx, GL_E_ARG, "gl_fri_layer_commit: NULL handle");
    *handle = nullptr;
    if (!is_pow2(len)) return fail(ctx, GL_E_ARG, "fri_committed_trees: length is not a power of two");
    unsigned lg = ilog2(len);
    if (arity_bits > lg || arity_bits > 8) return fail(ctx, GL_E_ARG, "fri_committed_trees: bad arity");
    if (cap_height > lg - arity_bits)
        return fail(ctx, GL_E_ARG, "MerkleTree::new: cap_height must be at most log2(leaves.len())");
    if (!values_ext) return fail(ctx, GL_E_ARG, "gl_fri_layer_commit: NULL buffer");
    TRY(check_device_ptr(ctx, space, values_ext, len * 16, "gl_fri_layer_commit: values_ext"));
    TRY(check_device_ptr(ctx, space, cap_out, (size_t)32 << cap_height, "gl_fri_layer_commit: cap_out"));
    Guard g(ctx);
    const u64* dv;
    TRY(stage_in(ctx, values_ext, len * 16, space, 0, &dv));
    std::unique_ptr<gl_commit> h;
    TRY(fri_tree_new(ctx, dv, lg, arity_bits, cap_height, &h));
    TRY(copy_out(ctx, cap_out, h->cap.get(), h->cap.bytes(), space));
    TRY(finish(ctx));
    *handle = h.release();
    return GL_OK;
}

extern "C" int gl_fri_fold(gl_ctx* ctx, const uint64_t* coeffs_ext, uint64_t len, uint32_t arity_bits,
                           const uint64_t beta[2], uint64_t shift, uint64_t* folded_coeffs_out,
                           uint64_t* next_values_out, int space) {
    if (!ctx) return GL_E_ARG;
    if (!is_pow2(len)) return fail(ctx, GL_E_ARG, "fri fold: length is not a power of two");
    unsigned lg = ilog2(len);
    if (arity_bits > lg) return fail(ctx, GL_E_ARG, "fri fold: arity larger than the polynomial");
    if (!coeffs_ext || !beta) return fail(ctx, GL_E_ARG, "gl_fri_fold: NULL buffer");
    TRY(check_device_ptr(ctx, space, coeffs_ext, len * 16, "gl_fri_fold: coeffs_ext"));
    TRY(check_device_ptr(ctx, space, folded_coeffs_out, (len >> arity_bits) * 16, "gl_fri_fold: folded_coeffs_out"));
    TRY(check_device_ptr(ctx, space, next_values_out, (len >> arity_bits) * 16, "gl_fri_fold: next_values_out"));
    Guard g(ctx);
    const u64* dcf;
    TRY(stage_in(ctx, coeffs_ext, len * 16, space, 0, &dcf));
    const u64 out_len = len >> arity_bits;
    const unsigned out_lg = lg - arity_bits;
    void *dcols, *dext;
    TRY(scratch_get(ctx, 2, out_len * 16, &dcols));
    TRY(scratch_get(ctx, 3, out_len * 16, &dext));
    launch_fri_fold(dcf, out_len, arity_bits, beta[0], beta[1], (u64*)dcols, out_len, ctx->stream);
    if (folded_coeffs_out) {
        u64* dst = space == GL_DEVICE ? folded_coeffs_out : (u64*)dext;
        launch_interleave2((const u64*)dcols, out_len, out_len, dst, ctx->stream);
        TRY(copy_out(ctx, folded_coeffs_out, dst, out_len * 16, space));
    }
    if (next_values_out) {
        u64 sh = glh::canon(shift);
        if (sh == 0) return fail(ctx, GL_E_ARG, "gl_fri_fold: zero coset shift");
        const u64* pre;
        TRY(pow_table(ctx, sh, &pre));
        TRY(transform_natural(ctx, (u64*)dcols, out_lg, 2, false, pre, nullptr));
        u64* dst = space == GL_DEVICE ? next_values_out : (u64*)dext;
        launch_interleave2((const u64*)dcols, out_len, out_len, dst, ctx->stream);
        TRY(copy_out(ctx, next_values_out, dst, out_len * 16, space));
    }
    return finish(ctx);
}

// prove_openings up to the FRI polynomial, everything left on the device: *d_coeffs / *d_values point into scratch
// slot 5 / 4 ([N][2] interleaved, natural order) and stay valid until the next call that uses those slots.
static int fri_final_poly_device(gl_ctx* ctx, gl_commit* const* oracles, uint32_t num_oracles, const gl_fri_batch* batches,
                                 uint32_t num_batches, const gl_fri_poly* polys, const uint64_t alpha[2], uint32_t rate_bits,
                                 bool times_x, bool want_values, u64** d_coeffs, u64** d_values) {
    if (!oracles || !num_oracles || !batches || !num_batches || !polys || !alpha)
        return fail(ctx, GL_E_ARG, "gl_fri_final_poly: NULL or empty argument");
    const uint32_t log_n = oracles[0]->log_n;
    for (uint32_t i = 0; i < num_oracles; i++) {
        if (!oracles[i] || oracles[i]->ctx != ctx || !oracles[i]->coeffs.get())
            return fail(ctx, GL_E_STATE, "gl_fri_final_poly: oracle is not a polynomial commit of this ctx");
        if (oracles[i]->log_n != log_n) return fail(ctx, GL_E_ARG, "gl_fri_final_poly: oracles of different degree");
    }
    if (log_n + rate_bits > 30) return fail(ctx, GL_E_ARG, "gl_fri_final_poly: log_n + rate_bits > 30 not supported");
    const u64 n = (u64)1 << log_n, N = n << rate_bits;
    uint32_t total = 0, kmax = 0;
    for (uint32_t b = 0; b < num_batches; b++) {
        if (batches[b].first_poly != total) return fail(ctx, GL_E_ARG, "gl_fri_final_poly: batches must tile polys[] in order");
        total += batches[b].num_polys;
        if (batches[b].num_polys > kmax) kmax = batches[b].num_polys;
        if (batches[b].num_polys == 0 || batches[b].num_polys > 2048)
            return fail(ctx, GL_E_ARG, "gl_fri_final_poly: a batch needs 1..2048 polynomials");
    }
    for (uint32_t j = 0; j < total; j++)
        if (polys[j].oracle_index >= num_oracles || polys[j].polynomial_index >= oracles[polys[j].oracle_index]->c)
            return fail(ctx, GL_E_ARG, "gl_fri_final_poly: polynomial index out of range");
    // scratch: 0 = pointer + power tables, 1 = transform scratch (transform_natural), 2 = composition poly,
    // 3 = final poly, 4 = padded columns then interleaved values, 5 = segment carries + interleaved coefficients
    void *d_tab, *d_comp, *d_final, *d_cols, *d_misc;
    const size_t tab_bytes = (size_t)kmax * (sizeof(u64*) + 16);
    TRY(scratch_get(ctx, 0, tab_bytes, &d_tab));
    TRY(scratch_get(ctx, 2, n * 16, &d_comp));
    TRY(scratch_get(ctx, 3, n * 16, &d_final));
    TRY(scratch_get(ctx, 4, N * 32, &d_cols));
    const size_t nseg = n / FRI_DIV_SEG + 1;
    TRY(scratch_get(ctx, 5, nseg * 32 + N * 16, &d_misc));
    u64* seg_h = (u64*)d_misc;
    u64* seg_b = seg_h + 2 * nseg;
    u64* d_ext = seg_b + 2 * nseg;
    CK(cudaMemsetAsync(d_final, 0, n * 16, ctx->stream));
    const glh::ext al = {glh::canon(alpha[0]), glh::canon(alpha[1])};
    std::vector<u64> host_tab;
    for (uint32_t b = 0; b < num_batches; b++) {
        const uint32_t k = batches[b].num_polys;
        host_tab.assign((size_t)k * 3, 0);
        glh::ext cur = {1, 0};
        for (uint32_t j = 0; j < k; j++) {
            const gl_fri_poly& fp = polys[batches[b].first_poly + j];
            host_tab[j] = (u64)(uintptr_t)(oracles[fp.oracle_index]->coeffs.get() + (size_t)fp.polynomial_index * n);
            host_tab[k + 2 * j] = cur.a;
            host_tab[k + 2 * j + 1] = cur.b;
            cur = glh::ext_mul(cur, al);
        }
        CK(cudaMemcpyAsync(d_tab, host_tab.data(), host_tab.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));   // host_tab is reused by the next batch
        launch_fri_reduce_polys((const u64* const*)d_tab, k, n, (const u64*)d_tab + k, (u64*)d_comp, ctx->stream);
        const glh::ext z = {glh::canon(batches[b].point[0]), glh::canon(batches[b].point[1])};
        const glh::ext zs = glh::ext_pow(z, FRI_DIV_SEG), sh = glh::ext_pow(al, k);
        const u64 zz[2] = {z.a, z.b}, zt[2] = {zs.a, zs.b}, shv[2] = {sh.a, sh.b};
        launch_fri_divide_accumulate((const u64*)d_comp, n, zz, zt, shv, seg_h, seg_b, (u64*)d_final, ctx->stream);
    }
    // final_poly.lde(rate_bits), then coset_fft(7) over the extension = two base transforms
    launch_ext_to_padded_cols((const u64*)d_final, n, N, (u64*)d_cols, d_ext, times_x ? 1 : 0, ctx->stream);
    *d_coeffs = d_ext;
    *d_values = nullptr;
    if (want_values) {
        const u64* pre;
        TRY(pow_table(ctx, 7, &pre));
        TRY(transform_natural(ctx, (u64*)d_cols, log_n + rate_bits, 2, false, pre, nullptr));
        u64* d_vals = (u64*)d_cols + 2 * N;
        launch_interleave2((const u64*)d_cols, N, N, d_vals, ctx->stream);
        *d_values = d_vals;
    }
    return GL_OK;
}

extern "C" int gl_fri_final_poly(gl_ctx* ctx, gl_commit* const* oracles, uint32_t num_oracles, const gl_fri_batch* batches,
                                 uint32_t num_batches, const gl_fri_poly* polys, const uint64_t alpha[2],
                                 uint32_t rate_bits, uint64_t* lde_coeffs_out, uint64_t* lde_values_out, int space) {
    if (!ctx) return GL_E_ARG;
    // both outputs are [N][2] extension elements, N >= 1: 16 bytes at least
    TRY(check_device_ptr(ctx, space, lde_coeffs_out, 16, "gl_fri_final_poly: lde_coeffs_out"));
    TRY(check_device_ptr(ctx, space, lde_values_out, 16, "gl_fri_final_poly: lde_values_out"));
    Guard g(ctx);
    u64 *dc, *dv;
    TRY(fri_final_poly_device(ctx, oracles, num_oracles, batches, num_batches, polys, alpha, rate_bits,
                              (ctx->compat & GL_COMPAT_FRI_FINAL_POLY_TIMES_X) != 0, lde_values_out != nullptr, &dc, &dv));
    const u64 N = ((u64)1 << oracles[0]->log_n) << rate_bits;
    TRY(copy_out(ctx, lde_coeffs_out, dc, N * 16, space));
    if (lde_values_out) TRY(copy_out(ctx, lde_values_out, dv, N * 16, space));
    return finish(ctx);
}

// ------------------------------------------------------------------------------------------------
// PolynomialBatch::prove_openings + fri_proof in ONE call (plonky2::fri::oracle / fri::prover): the FRI polynomial, the
// layer trees, the Fiat-Shamir sponge, the proof-of-work search and the query openings all stay on the device; the host
// synchronises three times (alpha, the PoW witness, the finished proof) instead of ~70 dependent round trips.
// ------------------------------------------------------------------------------------------------
extern "C" int gl_fri_proof_words(const gl_fri_params* prm, const uint32_t* oracle_columns, uint32_t num_oracles, uint32_t degree_bits,
                                  uint64_t* words_out) {
    if (!prm || !oracle_columns || !words_out || prm->num_reduction_layers > GL_FRI_MAX_LAYERS) return GL_E_ARG;
    const unsigned lgN = degree_bits + prm->rate_bits, h = prm->cap_height;
    if (h > lgN) return GL_E_ARG;
    uint64_t per_query = 1, words = 0;
    for (uint32_t i = 0; i < num_oracles; i++) per_query += oracle_columns[i] + 4ull * (lgN - h);
    unsigned lg = lgN;
    for (uint32_t l = 0; l < prm->num_reduction_layers; l++) {
        const unsigned ab = prm->reduction_arity_bits[l];
        if (ab == 0 || ab > 8 || ab > lg || h > lg - ab) return GL_E_ARG;
        words += 4ull << h;
        per_query += (2ull << ab) + 4ull * (lg - ab - h);
        lg -= ab;
    }
    if (lg < prm->rate_bits) return GL_E_ARG;
    words += 2ull << (lg - prm->rate_bits);   // final_poly
    words += 1;                               // pow_witness
    words += per_query * prm->num_query_rounds;
    *words_out = words;
    return GL_OK;
}

static int fri_params_check(gl_ctx* ctx, const gl_fri_params* prm, const char* name) {
    if (prm->num_reduction_layers > GL_FRI_MAX_LAYERS || prm->num_query_rounds == 0 || prm->num_query_rounds > 1024 ||
        prm->proof_of_work_bits > 48)
        return fail(ctx, GL_E_ARG, std::string(name) + ": unsupported FRI parameters");
    return GL_OK;
}

static int fri_prove_body(gl_ctx* ctx, gl_commit* const* oracles, uint32_t num_oracles, const gl_fri_batch* batches,
                          uint32_t num_batches, const gl_fri_poly* polys, const gl_fri_params* prm, gl_challenger* challenger,
                          uint64_t words, u64* d_proof, uint64_t* host_out, const u64* host_src, uint64_t host_words);

extern "C" int gl_fri_prove(gl_ctx* ctx, gl_commit* const* oracles, uint32_t num_oracles, const gl_fri_batch* batches,
                            uint32_t num_batches, const gl_fri_poly* polys, const gl_fri_params* prm, gl_challenger* challenger,
                            uint64_t* proof_out, uint64_t proof_cap_words, uint64_t* proof_words_out) {
    if (!ctx) return GL_E_ARG;
    if (!oracles || !num_oracles || !prm || !challenger || !proof_words_out)
        return fail(ctx, GL_E_ARG, "gl_fri_prove: NULL argument");
    if (challenger->input_len > 8 || challenger->output_len > 8) return fail(ctx, GL_E_ARG, "gl_fri_prove: bad challenger state");
    TRY(fri_params_check(ctx, prm, "gl_fri_prove"));
    for (uint32_t i = 0; i < num_oracles; i++)
        if (!oracles[i] || oracles[i]->ctx != ctx || !oracles[i]->coeffs.get() || !oracles[i]->finished || oracles[i]->shard_count != 1 ||
            oracles[i]->rate_bits != prm->rate_bits || oracles[i]->cap_height != prm->cap_height || oracles[i]->log_n != oracles[0]->log_n)
            return fail(ctx, GL_E_STATE, "gl_fri_prove: every oracle must be a finished, unsharded polynomial commit of this ctx with the FRI config's rate_bits / cap_height");
    std::vector<uint32_t> ocols(num_oracles);
    for (uint32_t i = 0; i < num_oracles; i++) ocols[i] = leaf_len(oracles[i]);
    uint64_t words = 0;
    if (gl_fri_proof_words(prm, ocols.data(), num_oracles, oracles[0]->log_n, &words) != GL_OK)
        return fail(ctx, GL_E_ARG, "gl_fri_prove: reduction_arity_bits do not fit the degree / cap_height");
    *proof_words_out = words;
    if (!proof_out || proof_cap_words < words) return fail(ctx, GL_E_ARG, "gl_fri_prove: proof buffer too small (see *proof_words_out)");
    Guard g(ctx);
    PoolBuf proof;
    TRY(proof.alloc(ctx, words * 8));
    return fri_prove_body(ctx, oracles, num_oracles, batches, num_batches, polys, prm, challenger, words, proof.get(), proof_out,
                          proof.get(), words);
}

// The body of gl_fri_prove, with the ctx held and the arguments checked: the proof's `words` words go to the device buffer
// d_proof, *challenger advances past the proof, and host_words words from host_src reach host_out with the final
// synchronisation (the proof itself, or a larger buffer that holds it).
static int fri_prove_body(gl_ctx* ctx, gl_commit* const* oracles, uint32_t num_oracles, const gl_fri_batch* batches,
                          uint32_t num_batches, const gl_fri_poly* polys, const gl_fri_params* prm, gl_challenger* challenger,
                          uint64_t words, u64* d_proof, uint64_t* host_out, const u64* host_src, uint64_t host_words) {
    const uint32_t degree_bits = oracles[0]->log_n, rate_bits = prm->rate_bits, h = prm->cap_height, rounds = prm->num_query_rounds;
    const unsigned lgN = degree_bits + rate_bits;
    const u64 N = (u64)1 << lgN;
    const uint32_t layers = prm->num_reduction_layers;
    // device state: challenger | alpha/beta scratch [2] | query challenges [rounds] | pow state [12] | pow best | response |
    // cumulative arity bits | query indices [(layers + 1)][rounds]
    PoolBuf state;
    TRY(state.alloc(ctx, (32 + 2 + rounds + 12 + 2 + GL_FRI_MAX_LAYERS + (size_t)(layers + 1) * rounds) * 8));
    u64* d_state = state.get();
    std::vector<std::unique_ptr<gl_commit>> trees;
    static_assert(sizeof(gl_challenger) == 29 * 8, "gl_challenger layout");
    gl_challenger* d_ch = (gl_challenger*)d_state;
    u64* d_ab = d_state + 32;
    u64* d_qch = d_ab + 2;
    u64* d_pow_state = d_qch + rounds;
    unsigned long long* d_best = (unsigned long long*)(d_pow_state + 12);
    u64* d_resp = d_pow_state + 13;
    uint32_t* d_cum = (uint32_t*)(d_pow_state + 14);
    u64* d_idx = d_pow_state + 14 + GL_FRI_MAX_LAYERS;
    CK(cudaMemcpyAsync(d_ch, challenger, sizeof(gl_challenger), cudaMemcpyHostToDevice, ctx->stream));
    // ---- alpha = challenger.get_extension_challenge(): the only challenge the host needs (power tables of the reduction)
    u64 alpha[2];
    launch_challenger_step(d_ch, nullptr, 0, d_ab, 2, nullptr, ctx->stream);
    CK(cudaMemcpyAsync(alpha, d_ab, 16, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    u64 *d_coeffs, *d_values;
    TRY(fri_final_poly_device(ctx, oracles, num_oracles, batches, num_batches, polys, alpha, rate_bits,
                              ((prm->flags | ctx->compat) & GL_COMPAT_FRI_FINAL_POLY_TIMES_X) != 0, true, &d_coeffs, &d_values));
    // ---- fri_committed_trees: per layer tree -> observe cap -> beta -> fold -> coset_fft, no host involvement
    u64 len = N;
    unsigned lg = lgN;
    u64 off = 0;                 // write position in the proof buffer
    u64 shift = 7;
    u64 *cur_coeffs = d_coeffs, *cur_values = d_values;
    PoolBuf folded_coeffs, folded_values;   // the previous layer's fold
    uint32_t cum[GL_FRI_MAX_LAYERS] = {}, acc_bits = 0;
    for (uint32_t l = 0; l < layers; l++) {
        const unsigned ab = prm->reduction_arity_bits[l];
        std::unique_ptr<gl_commit> t;
        TRY(fri_tree_new(ctx, cur_values, lg, ab, h, &t));
        CK(cudaMemcpyAsync(d_proof + off, t->cap.get(), t->cap.bytes(), cudaMemcpyDeviceToDevice, ctx->stream));
        off += 4ull << h;
        launch_challenger_step(d_ch, t->cap.get(), 4u << h, d_ab, 2, nullptr, ctx->stream);   // observe_cap, beta
        trees.push_back(std::move(t));
        shift = glh::pow(shift, (u64)1 << ab);
        const u64 out_len = len >> ab;
        PoolBuf n_coeffs, n_values;
        TRY(n_coeffs.alloc(ctx, out_len * 16));
        TRY(n_values.alloc(ctx, out_len * 16));
        void* dcols;
        TRY(scratch_get(ctx, 2, out_len * 16, &dcols));
        launch_fri_fold_dev(cur_coeffs, out_len, ab, d_ab, (u64*)dcols, out_len, ctx->stream);
        launch_interleave2((const u64*)dcols, out_len, out_len, n_coeffs.get(), ctx->stream);
        const u64* pre;
        TRY(pow_table(ctx, shift, &pre));
        TRY(transform_natural(ctx, (u64*)dcols, lg - ab, 2, false, pre, nullptr));
        launch_interleave2((const u64*)dcols, out_len, out_len, n_values.get(), ctx->stream);
        cur_coeffs = n_coeffs.get(); cur_values = n_values.get();
        folded_coeffs = std::move(n_coeffs);   // the fold before goes back to the pool: stream-ordered reuse
        folded_values = std::move(n_values);
        len = out_len; lg -= ab;
        acc_bits += ab;
        cum[l] = acc_bits;
    }
    // final_poly: "the coefficients being removed here are always zero"
    const u64 final_len = len >> rate_bits;
    CK(cudaMemcpyAsync(d_proof + off, cur_coeffs, final_len * 16, cudaMemcpyDeviceToDevice, ctx->stream));
    launch_challenger_step(d_ch, d_proof + off, (uint32_t)(2 * final_len), nullptr, 0, d_pow_state, ctx->stream);
    off += 2 * final_len;
    // ---- fri_proof_of_work: smallest witness; the input position is the number of pending inputs, which the host can count
    uint32_t pending = challenger->input_len;   // replay the buffer lengths of the transcript so far (values stay on the device)
    {
        auto observe = [&](uint64_t cnt) { pending = (uint32_t)((pending + cnt) % 8); };
        auto squeeze = [&]() { pending = 0; };
        squeeze();                                    // alpha
        for (uint32_t l = 0; l < layers; l++) { observe(4ull << h); squeeze(); }
        observe(2 * final_len);
    }
    const unsigned min_lz = prm->proof_of_work_bits;   // + (64 - F::order().bits()) = + 0
    const unsigned long long none = ~0ULL;
    CK(cudaMemcpyAsync(d_best, &none, 8, cudaMemcpyHostToDevice, ctx->stream));
    u64 witness = 0;
    {
        unsigned lg_chunk = min_lz + 2 < 14 ? 14 : (min_lz + 2 > 24 ? 24 : min_lz + 2);
        u64 chunk = (u64)1 << lg_chunk;
        bool found = false;
        for (u64 start = 0; start < GL_P && !found; start += chunk, chunk = chunk < ((u64)1 << 26) ? chunk * 2 : chunk) {
            u64 count = GL_P - start < chunk ? GL_P - start : chunk;
            launch_pow_grind(d_pow_state, pending, 7, min_lz, start, count, d_best, ctx->stream);
            unsigned long long best;
            CK(cudaMemcpyAsync(&best, d_best, 8, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            if (best != none) { witness = best; found = true; }
            else if (start >= ((u64)1 << 40)) break;
        }
        if (!found) return fail(ctx, GL_E_STATE, "fri_proof_of_work: no witness found");
    }
    // observe the witness, recompute the response with the normal Challenger code (as upstream does), then the query indices
    launch_challenger_step(d_ch, (const u64*)d_best, 1, d_resp, 1, nullptr, ctx->stream);
    CK(cudaMemcpyAsync(d_proof + off, d_best, 8, cudaMemcpyDeviceToDevice, ctx->stream));
    off += 1;
    launch_challenger_step(d_ch, nullptr, 0, d_qch, rounds, nullptr, ctx->stream);
    CK(cudaMemcpyAsync(d_cum, cum, sizeof cum, cudaMemcpyHostToDevice, ctx->stream));
    uint64_t query_stride = 1;
    for (uint32_t i = 0; i < num_oracles; i++) query_stride += leaf_len(oracles[i]) + 4ull * (lgN - h);
    for (auto& t : trees) query_stride += t->c + 4ull * (t->log_n - h);
    u64* d_queries = d_proof + off;
    launch_fri_query_indices(d_qch, rounds, lgN, d_cum, layers, d_idx, d_queries, query_stride, ctx->stream);
    u64 qoff = 1;
    for (uint32_t i = 0; i < num_oracles; i++) {
        const gl_commit* o = oracles[i];
        launch_gather_proof(o->lde.get(), o->n_local, leaf_len(o), o->digests.get(), lgN - h, d_idx, rounds, d_queries + qoff,
                            query_stride, ctx->stream);
        qoff += leaf_len(o) + 4ull * (lgN - h);
    }
    for (uint32_t l = 0; l < layers; l++) {
        const gl_commit* t = trees[l].get();
        launch_gather_proof(t->lde.get(), t->n_local, t->c, t->digests.get(), t->log_n - h, d_idx + (size_t)(l + 1) * rounds, rounds,
                            d_queries + qoff, query_stride, ctx->stream);
        qoff += t->c + 4ull * (t->log_n - h);
    }
    off += query_stride * rounds;
    if (off != words) return fail(ctx, GL_E_STATE, "gl_fri_prove: internal size mismatch");
    u64 response = 0;
    CK(cudaMemcpyAsync(host_out, host_src, host_words * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(challenger, d_ch, sizeof(gl_challenger), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&response, d_resp, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    if (min_lz && (response >> (64 - min_lz)) != 0)
        return fail(ctx, GL_E_STATE, "fri_proof_of_work: response does not have the required leading zeros");
    (void)witness;
    return GL_OK;
}

extern "C" int gl_ctx_set_compat(gl_ctx* ctx, uint32_t flags) {
    if (!ctx) return GL_E_ARG;
    if (flags & ~(uint32_t)GL_COMPAT_FRI_FINAL_POLY_TIMES_X) return fail(ctx, GL_E_ARG, "gl_ctx_set_compat: unknown flag");
    ctx->compat = flags;
    return GL_OK;
}

// ------------------------------------------------------------------------------------------------
// N3: compute_quotient_polys
// ------------------------------------------------------------------------------------------------
// The circuit geometry compute_quotient_polys supports (independent of the oracles)
static int quotient_geometry_check(gl_ctx* ctx, const gl_circuit* cd) {
    const uint32_t nch = cd->num_challenges, R = cd->num_routed_wires, deg = cd->quotient_degree_factor;
    if (nch == 0 || nch > QUOTIENT_MAX_CHALLENGES || cd->num_gates == 0 || cd->num_gates > QUOTIENT_MAX_GATES || R == 0 ||
        R > cd->num_wires || !is_pow2(deg) || cd->num_selectors == 0 || cd->num_selectors > cd->num_constants)
        return fail(ctx, GL_E_ARG, "gl_quotient_polys: unsupported circuit geometry");
    return GL_OK;
}
static int quotient_rate_check(gl_ctx* ctx, const gl_circuit* cd, uint32_t rate_bits) {
    const uint32_t qdb = ilog2(cd->quotient_degree_factor);
    if (qdb > rate_bits || qdb > 5)
        return fail(ctx, GL_E_ARG, "compute_quotient_polys: having constraints of degree higher than the rate is not supported");
    return GL_OK;
}
// gates[i] of a circuit that passed quotient_geometry_check
static int quotient_gate_check(gl_ctx* ctx, const gl_circuit* cd, const gl_gate& g, uint32_t i) {
    if (g.kind > GL_GATE_UNINTERLEAVE_TO_B32 || g.selector_index >= cd->num_selectors || g.group_start > i || g.group_end <= i ||
        g.group_end > cd->num_gates)
        return fail(ctx, GL_E_ARG, "gl_quotient_polys: bad gate descriptor");
    uint32_t need = 0;
    switch (g.kind) {
        case GL_GATE_CONSTANT: need = g.num_ops; if (cd->num_selectors + g.num_ops > cd->num_constants) need = ~0u; break;
        case GL_GATE_PUBLIC_INPUT: need = 4; break;
        case GL_GATE_U32_INTERLEAVE: need = g.num_ops * 34; break;
        case GL_GATE_UNINTERLEAVE_TO_U32:
        case GL_GATE_UNINTERLEAVE_TO_B32: need = g.num_ops * 67; break;
        default: break;
    }
    if (need > cd->num_wires) return fail(ctx, GL_E_ARG, "gl_quotient_polys: gate does not fit the wires / constants");
    return GL_OK;
}

// compute_quotient_polys with the ctx held (the body of gl_quotient_polys)
static int quotient_polys(gl_ctx* ctx, const gl_circuit* cd, const gl_gate* gates, const uint64_t* k_is,
                          gl_commit* constants_sigmas, gl_commit* wires, gl_commit* zs_pp, const uint64_t* public_inputs_hash,
                          const uint64_t* betas, const uint64_t* gammas, const uint64_t* alphas, uint64_t* chunks_out, int space) {
    if (!cd || !gates || !k_is || !constants_sigmas || !wires || !zs_pp || !public_inputs_hash || !betas || !gammas || !alphas ||
        !chunks_out)
        return fail(ctx, GL_E_ARG, "gl_quotient_polys: NULL argument");
    const uint32_t nch = cd->num_challenges, R = cd->num_routed_wires, deg = cd->quotient_degree_factor;
    TRY(quotient_geometry_check(ctx, cd));
    const uint32_t qdb = ilog2(deg), lg_n = cd->degree_bits;
    gl_commit* cm[3] = {constants_sigmas, wires, zs_pp};
    for (auto* h : cm) {
        if (h->ctx != ctx || !h->finished || !h->lde.get()) return fail(ctx, GL_E_STATE, "gl_quotient_polys: oracle is not a finished commit of this ctx");
        if (h->log_n != lg_n || h->rate_bits != wires->rate_bits) return fail(ctx, GL_E_ARG, "gl_quotient_polys: oracles of different degree or rate");
        if (h->shard_count != 1) return fail(ctx, GL_E_ARG, "gl_quotient_polys: sharded oracles are not supported");
    }
    const uint32_t rate_bits = wires->rate_bits;
    TRY(quotient_rate_check(ctx, cd, rate_bits));
    const uint32_t chunks = (R + deg - 1) / deg, num_prods = chunks - 1;
    if (constants_sigmas->c != cd->num_constants + R || wires->c != cd->num_wires || zs_pp->c != nch * chunks)
        return fail(ctx, GL_E_ARG, "gl_quotient_polys: column counts do not match the circuit description");
    quotient_args a;
    memset(&a, 0, sizeof a);
    uint32_t ngc = 0;
    for (uint32_t i = 0; i < cd->num_gates; i++) {
        const gl_gate& g = gates[i];
        TRY(quotient_gate_check(ctx, cd, g, i));
        a.gates[i] = g;
        ngc = std::max(ngc, quotient_gate_constraints(g));
    }
    const u64 n = (u64)1 << lg_n, lde_size = n << qdb;
    TRY(check_device_ptr(ctx, space, chunks_out, (size_t)nch * lde_size * 8, "gl_quotient_polys: chunks_out"));
    const uint32_t nterms = nch * (1 + chunks) + ngc;
    // tables: alpha powers [nch][nterms], k_is [R]
    std::vector<u64> tab((size_t)nch * nterms + R);
    for (uint32_t c = 0; c < nch; c++) {
        u64 cur = 1;
        const u64 al = glh::canon(alphas[c]);
        for (uint32_t t = 0; t < nterms; t++) {
            tab[(size_t)c * nterms + t] = cur;
            cur = glh::mul(cur, al);
        }
    }
    for (uint32_t j = 0; j < R; j++) tab[(size_t)nch * nterms + j] = glh::canon(k_is[j]);
    void *d_tab, *d_vals;
    TRY(scratch_get(ctx, 0, tab.size() * 8, &d_tab));
    TRY(scratch_get(ctx, 4, (size_t)nch * lde_size * 8, &d_vals));
    CK(cudaMemcpyAsync(d_tab, tab.data(), tab.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    const u64* xtab;
    TRY(pow_table(ctx, glh::root_of_unity(lg_n + qdb), &xtab));
    a.cs = constants_sigmas->lde.get(); a.cs_ld = constants_sigmas->n_local;
    a.wires = wires->lde.get(); a.w_ld = wires->n_local;
    a.zs = zs_pp->lde.get(); a.z_ld = zs_pp->n_local;
    a.lg_lde = lg_n + qdb; a.qdb = qdb; a.nch = nch; a.R = R; a.deg = deg; a.chunks = chunks; a.num_prods = num_prods;
    a.num_constants = cd->num_constants; a.num_selectors = cd->num_selectors; a.num_gates = cd->num_gates;
    a.nterms = nterms; a.gate_term0 = nch * (1 + chunks);
    a.apow = (const u64*)d_tab; a.k_is = (const u64*)d_tab + (size_t)nch * nterms; a.xtab = xtab;
    for (uint32_t c = 0; c < nch; c++) { a.betas[c] = glh::canon(betas[c]); a.gammas[c] = glh::canon(gammas[c]); }
    for (int i = 0; i < 4; i++) a.pih[i] = glh::canon(public_inputs_hash[i]);
    {   // ZeroPolyOnCoset::new(degree_bits, quotient_degree_bits): g^n w_rate^i - 1 and inverses
        const u64 g_pow_n = glh::pow(7, n), w_rate = glh::root_of_unity(qdb);
        u64 cur = 1;
        for (uint32_t i = 0; i < (1u << qdb); i++) {
            a.zh[i] = glh::sub(glh::mul(g_pow_n, cur), 1);
            a.zh_inv[i] = glh::inv(a.zh[i]);
            cur = glh::mul(cur, w_rate);
        }
    }
    a.n_field = glh::canon(n % GL_P);
    a.out = (u64*)d_vals;
    launch_quotient(a, ctx->stream);
    CK(cudaStreamSynchronize(ctx->stream));   // `tab` dies with this call; errors surface here
    // values.coset_ifft(F::coset_shift()) per challenge; the [nch][lde_size] result IS the chunk list
    const u64* post;
    TRY(pow_table(ctx, glh::inv(7), &post));
    TRY(transform_natural(ctx, (u64*)d_vals, lg_n + qdb, nch, true, nullptr, post));
    TRY(copy_out(ctx, chunks_out, d_vals, (size_t)nch * lde_size * 8, space));
    return finish(ctx);
}

extern "C" int gl_quotient_polys(gl_ctx* ctx, const gl_circuit* cd, const gl_gate* gates, const uint64_t* k_is,
                                 gl_commit* constants_sigmas, gl_commit* wires, gl_commit* zs_pp,
                                 const uint64_t* public_inputs_hash, const uint64_t* betas, const uint64_t* gammas,
                                 const uint64_t* alphas, uint64_t* chunks_out, int space) {
    if (!ctx) return GL_E_ARG;
    Guard g(ctx);
    return quotient_polys(ctx, cd, gates, k_is, constants_sigmas, wires, zs_pp, public_inputs_hash, betas, gammas, alphas,
                          chunks_out, space);
}

// ------------------------------------------------------------------------------------------------
// all_wires_permutation_partial_products: Z and the partial products, from the coefficients the two commits hold
// ------------------------------------------------------------------------------------------------
static int permutation_geometry_check(gl_ctx* ctx, const gl_circuit* cd) {
    const uint32_t nch = cd->num_challenges, R = cd->num_routed_wires, deg = cd->quotient_degree_factor;
    if (nch == 0 || nch > PERM_MAX_CHALLENGES || R == 0 || R > cd->num_wires || !is_pow2(deg))
        return fail(ctx, GL_E_ARG, "gl_permutation_zs: unsupported circuit geometry");
    if (nch * ((R + deg - 1) / deg) > PERM_MAX_SLOTS)
        return fail(ctx, GL_E_ARG, "gl_permutation_zs: num_challenges * ceil(num_routed_wires / quotient_degree_factor) > 64");
    return GL_OK;
}

// the body of gl_permutation_zs, with the ctx held
static int permutation_zs(gl_ctx* ctx, const gl_circuit* cd, const uint64_t* k_is, gl_commit* constants_sigmas, gl_commit* wires,
                          const uint64_t* betas, const uint64_t* gammas, uint64_t* zs_partial_products_out, int space,
                          uint64_t* grand_products_out) {
    if (!cd || !k_is || !constants_sigmas || !wires || !betas || !gammas || !zs_partial_products_out)
        return fail(ctx, GL_E_ARG, "gl_permutation_zs: NULL argument");
    if (space != GL_HOST && space != GL_DEVICE) return fail(ctx, GL_E_ARG, "gl_permutation_zs: bad space");
    const uint32_t nch = cd->num_challenges, R = cd->num_routed_wires, deg = cd->quotient_degree_factor;
    TRY(permutation_geometry_check(ctx, cd));
    const uint32_t chunks = (R + deg - 1) / deg;
    for (gl_commit* h : {constants_sigmas, wires}) {
        if (h->ctx != ctx || !h->finished || !h->coeffs.get())
            return fail(ctx, GL_E_STATE, "gl_permutation_zs: oracle is not a finished polynomial commit of this ctx");
        if (h->shard_count != 1) return fail(ctx, GL_E_ARG, "gl_permutation_zs: sharded oracles are not supported");
    }
    if (constants_sigmas->c != cd->num_constants + R || wires->c != cd->num_wires)
        return fail(ctx, GL_E_ARG, "gl_permutation_zs: column counts do not match the circuit description");
    if (wires->log_n != constants_sigmas->log_n || wires->log_n != cd->degree_bits)
        return fail(ctx, GL_E_ARG, "gl_permutation_zs: oracles of different degree");
    const uint32_t lg_n = cd->degree_bits;
    const u64 n = (u64)1 << lg_n;
    const size_t out_bytes = (size_t)nch * chunks * n * 8;
    TRY(check_device_ptr(ctx, space, zs_partial_products_out, out_bytes, "gl_permutation_zs: zs_partial_products_out"));
    const uint32_t nblocks = (uint32_t)((n + PERM_BLOCK - 1) / PERM_BLOCK);
    // small device state (scratch slot 0): k_is [R] | CTA products [nch][nblocks] | grand products [4] | zero flag
    std::vector<u64> kt(R);
    for (uint32_t j = 0; j < R; j++) kt[j] = glh::canon(k_is[j]);
    const size_t small_words = R + (size_t)nch * nblocks + PERM_MAX_CHALLENGES + 1;
    void* d_small;
    TRY(scratch_get(ctx, 0, small_words * 8, &d_small));
    u64* d_k = (u64*)d_small;
    u64* d_cta = d_k + R;
    u64* d_grand = d_cta + (size_t)nch * nblocks;
    unsigned* d_flag = (unsigned*)(d_grand + PERM_MAX_CHALLENGES);
    CK(cudaMemcpyAsync(d_k, kt.data(), R * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(d_flag, 0, sizeof(unsigned), ctx->stream));
    const u64* xtab;
    TRY(pow_table(ctx, glh::root_of_unity(lg_n), &xtab));
    void* d_out = zs_partial_products_out;
    if (space == GL_HOST) TRY(scratch_get(ctx, 4, out_bytes, &d_out));
    // the routed wire and sigma values: forward transforms of the coefficient columns (the salt of a blinded commit
    // lives only in its leaves).  The transforms run through scratch slot 1.
    PoolBuf rec;
    TRY(rec.alloc(ctx, (size_t)2 * R * n * 8));
    u64* d_rec = rec.get();
    TRY(transform_natural(ctx, d_rec, lg_n, R, false, nullptr, nullptr, wires->coeffs.get()));
    TRY(transform_natural(ctx, d_rec + (size_t)R * n, lg_n, R, false, nullptr, nullptr,
                          constants_sigmas->coeffs.get() + (size_t)cd->num_constants * n));
    perm_args a;
    memset(&a, 0, sizeof a);
    a.wires = d_rec; a.sigmas = d_rec + (size_t)R * n; a.k_is = d_k; a.xtab = xtab;
    a.out = (u64*)d_out; a.cta = d_cta; a.grand = d_grand; a.zero_den = d_flag;
    a.n = n; a.R = R; a.deg = deg; a.chunks = chunks; a.nch = nch; a.nblocks = nblocks;
    for (uint32_t c = 0; c < nch; c++) { a.betas[c] = glh::canon(betas[c]); a.gammas[c] = glh::canon(gammas[c]); }
    cudaError_t e = launch_permutation_zs(a, ctx->stream);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "launch_permutation_zs");
    u64 grand[PERM_MAX_CHALLENGES];
    unsigned zero_den = 0;
    e = cudaMemcpyAsync(grand, d_grand, nch * 8, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&zero_den, d_flag, sizeof zero_den, cudaMemcpyDeviceToHost, ctx->stream);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "download grand products");
    if (space == GL_HOST) TRY(copy_out(ctx, zs_partial_products_out, d_out, out_bytes, GL_HOST));
    TRY(finish(ctx));
    if (zero_den)
        return fail(ctx, GL_E_ARG, "gl_permutation_zs: wire + beta * sigma + gamma is zero at some row "
                                   "(batch_multiplicative_inverse of a zero denominator)");
    if (grand_products_out)
        for (uint32_t c = 0; c < nch; c++) grand_products_out[c] = grand[c];
    return GL_OK;
}

extern "C" int gl_permutation_zs(gl_ctx* ctx, const gl_circuit* cd, const uint64_t* k_is, gl_commit* constants_sigmas,
                                 gl_commit* wires, const uint64_t* betas, const uint64_t* gammas,
                                 uint64_t* zs_partial_products_out, int space, uint64_t* grand_products_out) {
    if (!ctx) return GL_E_ARG;
    Guard g(ctx);
    return permutation_zs(ctx, cd, k_is, constants_sigmas, wires, betas, gammas, zs_partial_products_out, space,
                          grand_products_out);
}

// ------------------------------------------------------------------------------------------------
// plonky2::plonk::prover::prove from the witness on: the stages above chained by the Fiat-Shamir transcript
// ------------------------------------------------------------------------------------------------
// The prover's three commits; they die (back to the pool) when gl_prove returns, on every path.
struct ProveOracles {
    std::unique_ptr<gl_commit> wires, zs, quotient;
};

// Pops `n` challenges from the device challenger into host memory (one small copy and a synchronisation).
static int draw_challenges(gl_ctx* ctx, gl_challenger* d_ch, const u64* observe, uint32_t n_obs, u64* d_out, uint32_t n,
                           u64* host_out) {
    launch_challenger_step(d_ch, observe, n_obs, d_out, n, nullptr, ctx->stream);
    CK(cudaMemcpyAsync(host_out, d_out, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    return finish(ctx);
}

static int prove_body(gl_ctx* ctx, const gl_circuit* cd, const gl_gate* gates, const uint64_t* k_is, gl_commit* cs,
                      const uint64_t circuit_digest[4], const gl_fri_params* prm, const HostCols& witness, int space,
                      const uint64_t* public_inputs, uint32_t num_public_inputs, uint64_t* proof_out, uint64_t fri_words,
                      uint64_t total_words, ProveOracles& o) {
    const uint32_t lg_n = cd->degree_bits, nch = cd->num_challenges, R = cd->num_routed_wires, qdf = cd->quotient_degree_factor;
    const uint32_t rate_bits = prm->rate_bits, h = prm->cap_height, zcols = nch * ((R + qdf - 1) / qdf), qcols = nch * qdf;
    const u64 n = (u64)1 << lg_n, cap_words = 4ull << h;
    // the proof as it goes back: caps [3][2^h][4] | OpeningSet | FRI proof
    PoolBuf out, st;
    TRY(out.alloc(ctx, total_words * 8));
    u64* d_caps = out.get();
    u64* d_open = d_caps + 3 * cap_words;
    u64* d_cs_open = d_open;                                   // constants | plonk_sigmas
    u64* d_w_open = d_cs_open + 2 * (size_t)cs->c;             // wires
    u64* d_z_open = d_w_open + 2 * (size_t)cd->num_wires;      // plonk_zs
    u64* d_znext_open = d_z_open + 2 * (size_t)nch;            // plonk_zs_next
    u64* d_pp_open = d_znext_open + 2 * (size_t)nch;           // partial_products
    u64* d_q_open = d_pp_open + 2 * (size_t)(zcols - nch);     // quotient_polys
    u64* d_fri = d_q_open + 2 * (size_t)qcols;
    // transcript state: challenger [32] | circuit digest [4] | public-inputs hash [4] | challenges [max(2 nch, 2)] | public inputs
    static_assert(sizeof(gl_challenger) == 29 * 8, "gl_challenger layout");
    TRY(st.alloc(ctx, (32 + 8 + 2 * (size_t)nch + 2 + num_public_inputs) * 8));
    gl_challenger* d_ch = (gl_challenger*)st.get();
    u64* d_digest = st.get() + 32;
    u64* d_pih = d_digest + 4;
    u64* d_chal = d_pih + 4;
    u64* d_pi = d_chal + 2 * (size_t)nch + 2;
    CK(cudaMemsetAsync(d_ch, 0, sizeof(gl_challenger), ctx->stream));   // Challenger::new()
    CK(cudaMemcpyAsync(d_digest, circuit_digest, 32, cudaMemcpyHostToDevice, ctx->stream));
    if (num_public_inputs)
        CK(cudaMemcpyAsync(d_pi, public_inputs, (size_t)num_public_inputs * 8, cudaMemcpyHostToDevice, ctx->stream));
    launch_hash_no_pad_rows(d_pi, num_public_inputs, 1, d_pih, ctx->stream);   // no inputs: [0, 0, 0, 0]
    // wires commit, then observe digest, pih, wires cap and draw betas, gammas
    TRY(commit_make(ctx, witness, true, lg_n, cd->num_wires, rate_bits, h, HostCols(), nullptr, space, "gl_prove: wires commit",
                    false, &o.wires));
    CK(cudaMemcpyAsync(d_caps, o.wires->cap.get(), cap_words * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    launch_challenger_step(d_ch, d_digest, 8, nullptr, 0, nullptr, ctx->stream);
    std::vector<u64> bg(2 * (size_t)nch + 4);
    u64 *betas = bg.data(), *gammas = betas + nch, *pih = gammas + nch;
    CK(cudaMemcpyAsync(pih, d_pih, 32, cudaMemcpyDeviceToHost, ctx->stream));
    TRY(draw_challenges(ctx, d_ch, d_caps, (uint32_t)cap_words, d_chal, 2 * nch, betas));
    // Z and the partial products, resident, and their commit; observe the cap, draw alphas
    {
        PoolBuf zs;
        TRY(zs.alloc(ctx, (size_t)zcols * n * 8));
        TRY(permutation_zs(ctx, cd, k_is, cs, o.wires.get(), betas, gammas, zs.get(), GL_DEVICE, nullptr));
        HostCols zin;
        zin.flat = zs.get();
        TRY(commit_make(ctx, zin, true, lg_n, zcols, rate_bits, h, HostCols(), nullptr, GL_DEVICE, "gl_prove: Z commit", false, &o.zs));
    }
    CK(cudaMemcpyAsync(d_caps + cap_words, o.zs->cap.get(), cap_words * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    std::vector<u64> alphas(nch);
    TRY(draw_challenges(ctx, d_ch, d_caps + cap_words, (uint32_t)cap_words, d_chal, nch, alphas.data()));
    // the quotient chunks, resident, and their commit; observe the cap, draw zeta
    {
        PoolBuf q;
        TRY(q.alloc(ctx, (size_t)qcols * n * 8));
        TRY(quotient_polys(ctx, cd, gates, k_is, cs, o.wires.get(), o.zs.get(), pih, betas, gammas, alphas.data(), q.get(), GL_DEVICE));
        HostCols qin;
        qin.flat = q.get();
        TRY(commit_make(ctx, qin, false, lg_n, qcols, rate_bits, h, HostCols(), nullptr, GL_DEVICE, "gl_prove: quotient commit", false,
                        &o.quotient));
    }
    CK(cudaMemcpyAsync(d_caps + 2 * cap_words, o.quotient->cap.get(), cap_words * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    u64 zeta[2];
    TRY(draw_challenges(ctx, d_ch, d_caps + 2 * cap_words, (uint32_t)cap_words, d_chal, 2, zeta));
    const glh::ext z = {zeta[0], zeta[1]};
    const glh::ext zn = glh::ext_pow(z, n);
    if (zn.a == 1 && zn.b == 0)
        return fail(ctx, GL_E_STATE, "gl_prove: Opening point is in the subgroup.");
    const glh::ext gz = glh::ext_mul(z, glh::ext{glh::root_of_unity(lg_n), 0});
    const u64 zeta_next[2] = {gz.a, gz.b};
    // OpeningSet::new, written in place in the proof buffer
    TRY(commit_eval(ctx, cs, 0, cs->c, zeta, d_cs_open, GL_DEVICE));
    TRY(commit_eval(ctx, o.wires.get(), 0, o.wires->c, zeta, d_w_open, GL_DEVICE));
    TRY(commit_eval(ctx, o.zs.get(), 0, nch, zeta, d_z_open, GL_DEVICE));
    TRY(commit_eval(ctx, o.zs.get(), 0, nch, zeta_next, d_znext_open, GL_DEVICE));
    if (zcols > nch) TRY(commit_eval(ctx, o.zs.get(), nch, zcols - nch, zeta, d_pp_open, GL_DEVICE));
    TRY(commit_eval(ctx, o.quotient.get(), 0, qcols, zeta, d_q_open, GL_DEVICE));
    // observe_openings(to_fri_openings()): [constants, plonk_sigmas, wires, plonk_zs, partial_products, quotient_polys], then
    // [plonk_zs_next]
    launch_challenger_step(d_ch, d_open, (uint32_t)(d_znext_open - d_open), nullptr, 0, nullptr, ctx->stream);
    launch_challenger_step(d_ch, d_pp_open, (uint32_t)(d_fri - d_pp_open), nullptr, 0, nullptr, ctx->stream);
    launch_challenger_step(d_ch, d_znext_open, 2 * nch, nullptr, 0, nullptr, ctx->stream);
    gl_challenger ch;
    CK(cudaMemcpyAsync(&ch, d_ch, sizeof ch, cudaMemcpyDeviceToHost, ctx->stream));
    TRY(finish(ctx));
    // prove_openings over get_fri_instance(zeta): every polynomial at zeta, the Z polynomials at g * zeta
    gl_commit* oracles[4] = {cs, o.wires.get(), o.zs.get(), o.quotient.get()};
    std::vector<gl_fri_poly> polys;
    for (uint32_t i = 0; i < 4; i++)
        for (uint32_t j = 0; j < oracles[i]->c; j++) polys.push_back({i, j});
    const uint32_t at_zeta = (uint32_t)polys.size();
    for (uint32_t j = 0; j < nch; j++) polys.push_back({2, j});
    gl_fri_batch batches[2] = {{{zeta[0], zeta[1]}, 0, at_zeta}, {{zeta_next[0], zeta_next[1]}, at_zeta, nch}};
    return fri_prove_body(ctx, oracles, 4, batches, 2, polys.data(), prm, &ch, fri_words, d_fri, proof_out, out.get(), total_words);
}

extern "C" int gl_prove(gl_ctx* ctx, const gl_circuit* cd, const gl_gate* gates, const uint64_t* k_is, gl_commit* constants_sigmas,
                        const uint64_t circuit_digest[4], const gl_fri_params* prm, const uint64_t* wires,
                        const uint64_t* const* wires_cols, int space, const uint64_t* public_inputs, uint32_t num_public_inputs,
                        uint64_t* proof_out, uint64_t proof_cap_words, uint64_t* proof_words_out) {
    if (!ctx) return GL_E_ARG;
    if (!cd || !gates || !k_is || !constants_sigmas || !circuit_digest || !prm || !proof_words_out ||
        (num_public_inputs && !public_inputs))
        return fail(ctx, GL_E_ARG, "gl_prove: NULL argument");
    if ((wires != nullptr) == (wires_cols != nullptr))
        return fail(ctx, GL_E_ARG, "gl_prove: pass the witness either as one array or as one array per wire");
    if ((space != GL_HOST && space != GL_DEVICE) || (wires_cols && space != GL_HOST))
        return fail(ctx, GL_E_ARG, "gl_prove: bad space (per-wire arrays are host memory)");
    const gl_commit* cs = constants_sigmas;
    const uint32_t nch = cd->num_challenges, R = cd->num_routed_wires, qdf = cd->quotient_degree_factor;
    // every geometry check of the two stage calls, before any work is done
    TRY(permutation_geometry_check(ctx, cd));
    TRY(quotient_geometry_check(ctx, cd));
    TRY(quotient_rate_check(ctx, cd, prm->rate_bits));
    for (uint32_t i = 0; i < cd->num_gates; i++) TRY(quotient_gate_check(ctx, cd, gates[i], i));
    if (ctx->shard_count != 1) return fail(ctx, GL_E_ARG, "gl_prove: sharded proving is not supported");
    if (cs->ctx != ctx || !cs->finished || !cs->coeffs.get() || cs->salt || cs->shard_count != 1)
        return fail(ctx, GL_E_ARG, "gl_prove: constants_sigmas must be a finished, unblinded, unsharded polynomial commit of this ctx");
    if (cs->log_n != cd->degree_bits || cs->c != cd->num_constants + R)
        return fail(ctx, GL_E_ARG, "gl_prove: constants_sigmas does not have the circuit's degree and num_constants + num_routed_wires columns");
    if (cs->rate_bits != prm->rate_bits || cs->cap_height != prm->cap_height)
        return fail(ctx, GL_E_ARG, "gl_prove: the FRI config's rate_bits / cap_height differ from constants_sigmas'");
    TRY(fri_params_check(ctx, prm, "gl_prove"));
    const uint32_t zcols = nch * ((R + qdf - 1) / qdf), qcols = nch * qdf;
    const uint32_t ocols[4] = {cs->c, cd->num_wires, zcols, qcols};
    uint64_t fri_words = 0;
    if (gl_fri_proof_words(prm, ocols, 4, cd->degree_bits, &fri_words) != GL_OK)
        return fail(ctx, GL_E_ARG, "gl_prove: reduction_arity_bits do not fit the degree / cap_height");
    const uint64_t total = 3 * (4ull << prm->cap_height) + 2ull * (cs->c + cd->num_wires + 2 * nch + (zcols - nch) + qcols) + fri_words;
    *proof_words_out = total;
    if (!proof_out || proof_cap_words < total) return fail(ctx, GL_E_ARG, "gl_prove: proof buffer too small (see *proof_words_out)");
    TRY(check_device_ptr(ctx, space, wires, ((size_t)cd->num_wires << cd->degree_bits) * 8, "gl_prove: wires"));
    Guard g(ctx);
    HostCols witness;
    witness.flat = const_cast<uint64_t*>(wires);
    witness.cols = const_cast<uint64_t* const*>(wires_cols);
    ProveOracles o;
    int rc = prove_body(ctx, cd, gates, k_is, constants_sigmas, circuit_digest, prm, witness, space, public_inputs, num_public_inputs,
                        proof_out, fri_words, total, o);
    if (rc != GL_OK) quiesce(ctx);   // nothing of a failed call is still running when its commits go back to the pool
    return rc;
}

extern "C" int gl_pow_grind(gl_ctx* ctx, const uint64_t state[12], uint32_t input_pos, uint32_t min_leading_zeros,
                            uint64_t* witness_out) {
    if (!ctx) return GL_E_ARG;
    if (!state || !witness_out || input_pos >= 12 || min_leading_zeros > 64)
        return fail(ctx, GL_E_ARG, "gl_pow_grind: bad argument");
    Guard g(ctx);
    void* d;
    TRY(scratch_get(ctx, 0, 13 * 8, &d));
    u64* dstate = (u64*)d;
    unsigned long long* dbest = (unsigned long long*)(dstate + 12);
    unsigned long long none = ~0ULL;
    CK(cudaMemcpyAsync(dstate, state, 96, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dbest, &none, 8, cudaMemcpyHostToDevice, ctx->stream));
    // The first batch holds four times the expected number of tries (it finds a witness with probability
    // 1 - e^-4); later batches double.  Batches are scanned in order and each keeps its minimum, so the
    // result is the smallest witness whatever the batch sizes.
    unsigned lg_chunk = min_leading_zeros + 2 < 14 ? 14 : (min_leading_zeros + 2 > 24 ? 24 : min_leading_zeros + 2);
    u64 chunk = (u64)1 << lg_chunk;
    // witnesses are field elements: upstream searches 0 .. p-1
    for (u64 start = 0; start < GL_P; start += chunk, chunk = chunk < ((u64)1 << 26) ? chunk * 2 : chunk) {
        u64 count = GL_P - start < chunk ? GL_P - start : chunk;
        launch_pow_grind(dstate, input_pos, 7, min_leading_zeros, start, count, dbest, ctx->stream);
        unsigned long long best;
        CK(cudaMemcpyAsync(&best, dbest, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (best != none) {
            *witness_out = best;
            return GL_OK;
        }
        if (start >= ((u64)1 << 40)) break;  // 2^40 failed candidates: min_leading_zeros is unreasonable
    }
    return fail(ctx, GL_E_STATE, "gl_pow_grind: no witness found");
}

// multi-GPU plane (NCCL behind the C ABI)
#include "gl_group.inc.cu"
