// spb_api.cu -- implementation of the C ABI declared in include/spsparse_b200.h.
// Host orchestration only; every data-path step is one of the hand-written kernels in
// radix_sort.cuh / reduce_by_key.cuh / scan.cuh / csr.cuh / spgemm.cuh / gen.cuh.  No CUB, Thrust,
// cuSPARSE or CPU fallback.
#include "../../include/spsparse_b200.h"

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <map>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <vector>

#include "common.cuh"
#include "csr.cuh"
#include "gen.cuh"
#include "radix_sort.cuh"
#include "radix_sort9.cuh"
#include "reduce_by_key.cuh"
#include "reduce_segsort.cuh"
#include "reduce_warp.cuh"
#include "scan.cuh"
#include "spgemm.cuh"
#include "dense_ops.cuh"
#include "rowpart.cuh"
#include "cons_plan.cuh"
#include "mm_pattern.cuh"

thread_local std::string g_last_error;

int spb_fail(int code, const char *fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

static inline double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
static double g_alloc_ms = 0;   // host time spent inside cudaMallocAsync (SPB_TRACE diagnostics)
static int g_trace = -1;
static inline bool tracing() {
    if (g_trace < 0) g_trace = getenv("SPB_TRACE") ? 1 : 0;
    return g_trace == 1;
}

// ---- device memory pool ----------------------------------------------------------------------------
// A size-keyed cache of cudaMalloc'ed blocks.  The hot path asks for the same multi-GB sizes every
// call; the driver's stream-ordered pool re-maps physical memory for them again and again (20-350 ms
// per request measured on B200), so blocks are kept here and handed back on an (almost) exact size
// match.  All use is ordered on the context's single stream, so a freed block can be reused at once.
struct DevPool {
    std::multimap<size_t, void *> free_;
    std::unordered_map<void *, size_t> live_;
    std::mutex mu_;
    size_t cached_bytes = 0;
    // SPB_POOL_POISON (tests): every block handed out is first filled with this byte over its whole size, on `stream`, so a
    // kernel that reads a slot nobody wrote sees the pattern instead of zeros or the previous call's data; -1 = off
    int poison = -1;
    cudaStream_t stream = nullptr;

    static size_t round_up(size_t b) {
        if (b < 512) return 512;
        if (b < (1u << 20)) return (b + 511) & ~(size_t)511;
        return (b + (1u << 20) - 1) & ~(size_t)((1u << 20) - 1);
    }
    cudaError_t alloc(void **out, size_t bytes) {
        std::lock_guard<std::mutex> g(mu_);
        const size_t want = round_up(bytes);
        auto it = free_.lower_bound(want);
        // at most 12.5% slack -- 50% for blocks of 64 MB and more: the panels of a row-panel multiply ask for a different
        // multi-GB size every time, and a cudaMalloc of that size stalls the stream for milliseconds
        if (it != free_.end() && it->first <= want + (want >= (64u << 20) ? want / 2 : want / 8)) {
            *out = it->second;
            live_[*out] = it->first;
            cached_bytes -= it->first;
            const size_t got = it->first;
            free_.erase(it);
            return poison >= 0 ? cudaMemsetAsync(*out, poison, got, stream) : cudaSuccess;
        }
        void *p = nullptr;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {  // give cached blocks back to the driver and retry once
            cudaGetLastError();
            trim_locked();
            e = cudaMalloc(&p, want);
            if (e != cudaSuccess) return e;
        }
        live_[p] = want;
        *out = p;
        return poison >= 0 ? cudaMemsetAsync(p, poison, want, stream) : cudaSuccess;
    }
    void release(void *p) {
        if (!p) return;
        std::lock_guard<std::mutex> g(mu_);
        auto it = live_.find(p);
        if (it == live_.end()) return;  // not ours (wrapped caller memory)
        free_.insert({it->second, p});
        cached_bytes += it->second;
        live_.erase(it);
    }
    void trim_locked() {
        cudaDeviceSynchronize();
        for (auto &kv : free_) cudaFree(kv.second);
        free_.clear();
        cached_bytes = 0;
    }
    void destroy() {
        std::lock_guard<std::mutex> g(mu_);
        trim_locked();
        for (auto &kv : live_) cudaFree(kv.first);
        live_.clear();
    }
};

struct spb_ctx {
    int device;
    cudaStream_t stream;
    bool own_stream;
    int sm_count;
    u32 merge_max_products;  // bin threshold, env SPB_MERGE_MAX_PRODUCTS
    u64 esc_chunk;           // products per expand-sort-compress chunk, env SPB_ESC_CHUNK
    u64 hash_min_products;   // long rows with at least this many products use the bitmap + hash-accumulator kernels; ~0 = never (SPB_HASH_MIN_PRODUCTS)
    int hash_variant;        // 0: 1024 threads x 10240 outputs per item, 1: 512 x 5120 (two blocks per SM), 2: 256 x 2560 (four)  (SPB_HASH_VARIANT)
    u64 launches;            // kernels launched so far (bench.py reports it as gpu_launches)
    bool bulk_load;          // radix passes after the first bring their tile in with cp.async.bulk (SPB_BULK_LOAD, default on)
    // pageable host memory <-> device: worker threads copy through pinned staging buffers (see staged_copy)
    static constexpr int XFER_WORKERS = 8;   // at most; xfer_workers of them are used (SPB_XFER_WORKERS, default: half the host's threads)
    int xfer_workers;
    static constexpr size_t XFER_CHUNK = 16u << 20;
    void *xfer_buf[XFER_WORKERS][2];
    cudaStream_t xfer_stream[XFER_WORKERS];
    cudaEvent_t xfer_ev[XFER_WORKERS][2];
    bool xfer_ready;
    DevPool pool;
};

struct spb_coo {
    int rank;
    u64 shape[2];
    u64 n;
    i32 *idx[2];
    double *val;
    int sort_order[2];
    bool owned;
    // lazily cached structure of a sorted array (the reference caches dim_beginnings the same way,
    // VectorCooArray.hpp:323-335); valid for leading dimension sort_order[0]
    u32 *row_start;  // [nrows+1] compressed row starts incl. sentinel
    i32 *row_id;     // [nrows]
    u32 nrows;
    bool rows_valid;
    u32 *dense_ptr;  // [extent+1] dense pointer over the leading index, or nullptr
    bool dense_ptr_owned;
    u32 *range_ptr;  // [1 + (hi-lo) + 1] scan behind spb_coo_dense_ptr_range (its answer starts at range_ptr + 1), or nullptr
    u64 range_lo, range_hi;
    u32 max_row_len;  // longest compressed row, 0 = not computed yet (cached with the row structure)
};

// ---- stream-ordered scratch memory, released when the scope ends ---------------------------------
struct Scratch {
    spb_ctx *ctx;
    std::vector<void *> ptrs;
    explicit Scratch(spb_ctx *c) : ctx(c) {}
    ~Scratch() { for (void *p : ptrs) ctx->pool.release(p); }
    template <typename T>
    int get(T **out, u64 count) {
        void *p = nullptr;
        size_t bytes = (size_t)(count ? count : 1) * sizeof(T);
        double t0 = tracing() ? now_ms() : 0;
        cudaError_t e = ctx->pool.alloc(&p, bytes);
        if (tracing()) { double dt = now_ms() - t0; g_alloc_ms += dt; if (dt > 1.0) fprintf(stderr, "[spb] pool.alloc(%zu MB) took %.2f ms\n", bytes >> 20, dt); }
        if (e != cudaSuccess) return spb_fail(SPB_ERR_CUDA, "device allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
        ptrs.push_back(p);
        *out = (T *)p;
        return 0;
    }
    template <typename T>
    int zeroed(T **out, u64 count) {
        CKR(get(out, count));
        CK(cudaMemsetAsync(*out, 0, (size_t)(count ? count : 1) * sizeof(T), ctx->stream));
        return 0;
    }
    void release(void *p) {  // free early
        for (size_t i = 0; i < ptrs.size(); ++i)
            if (ptrs[i] == p) { ctx->pool.release(p); ptrs.erase(ptrs.begin() + i); return; }
    }
    void keep(void *p) {  // hand ownership to the caller
        for (size_t i = 0; i < ptrs.size(); ++i)
            if (ptrs[i] == p) { ptrs.erase(ptrs.begin() + i); return; }
    }
};

struct Timer {  // CUDA events on the context stream
    cudaStream_t s;
    std::vector<cudaEvent_t> ev;
    explicit Timer(cudaStream_t st) : s(st) {}
    ~Timer() { for (auto e : ev) cudaEventDestroy(e); }
    int mark() {
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, s);
        ev.push_back(e);
        return (int)ev.size() - 1;
    }
    float ms(int a, int b) {
        float t = 0;
        cudaEventSynchronize(ev[b]);
        cudaEventElapsedTime(&t, ev[a], ev[b]);
        return t;
    }
};

static inline u32 grid_for(u64 n, u32 threads, u32 cap) {
    u64 g = div_up(n ? n : 1, threads);
    return (u32)(g < cap ? g : cap);
}

// ---- host <-> device transfers of caller memory -----------------------------------------------------------------------
// A reference user's arrays are std::vectors: pageable memory, which the driver can only move through its own single
// staging pipeline (6-10 GB/s measured).  Here xfer_workers threads (up to XFER_WORKERS) each copy every xfer_workers-th chunk between the
// caller's memory and a pinned double buffer of their own and move it with an asynchronous copy on their own stream, so
// the CPU-side copies of several chunks and the DMA transfers overlap.  Pinned (or registered) caller memory is moved
// directly.  Synchronous for the caller, as the C ABI promises.
static bool host_ptr_is_pinned(const void *p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
}

static int xfer_setup(spb_ctx *c) {
    if (c->xfer_ready) return 0;
    {
        int want = getenv("SPB_XFER_WORKERS") ? atoi(getenv("SPB_XFER_WORKERS")) : (int)(std::thread::hardware_concurrency() / 2);
        c->xfer_workers = want < 1 ? 1 : (want > spb_ctx::XFER_WORKERS ? spb_ctx::XFER_WORKERS : want);
    }
    for (int w = 0; w < c->xfer_workers; ++w) {
        CK(cudaStreamCreateWithFlags(&c->xfer_stream[w], cudaStreamNonBlocking));
        for (int b = 0; b < 2; ++b) {
            CK(cudaHostAlloc(&c->xfer_buf[w][b], spb_ctx::XFER_CHUNK, cudaHostAllocDefault));
            CK(cudaEventCreateWithFlags(&c->xfer_ev[w][b], cudaEventDisableTiming));
        }
    }
    c->xfer_ready = true;
    return 0;
}

struct XferJob { void *dev; void *host; size_t bytes; };   // one array

// to_device: host -> dev, else dev -> host.  The device side must be complete / consumable on ctx->stream order: the
// caller synchronises ctx->stream before (downloads) -- uploads land before this returns.
static int staged_copy(spb_ctx *c, const XferJob *jobs, int njobs, bool to_device) {
    // pinned caller memory: plain asynchronous copies
    bool all_pinned = true;
    size_t total = 0;
    for (int j = 0; j < njobs; ++j) { if (jobs[j].bytes) { all_pinned = all_pinned && host_ptr_is_pinned(jobs[j].host); total += jobs[j].bytes; } }
    if (all_pinned || total < (4u << 20)) {
        for (int j = 0; j < njobs; ++j)
            if (jobs[j].bytes)
                CK(cudaMemcpyAsync(to_device ? jobs[j].dev : jobs[j].host, to_device ? jobs[j].host : jobs[j].dev, jobs[j].bytes,
                                   to_device ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        return 0;
    }
    CKR(xfer_setup(c));
    // the chunk list over all arrays
    struct Chunk { char *dev; char *host; size_t bytes; };
    std::vector<Chunk> chunks;
    for (int j = 0; j < njobs; ++j)
        for (size_t o = 0; o < jobs[j].bytes; o += spb_ctx::XFER_CHUNK)
            chunks.push_back({(char *)jobs[j].dev + o, (char *)jobs[j].host + o, std::min(spb_ctx::XFER_CHUNK, jobs[j].bytes - o)});
    const int NW = c->xfer_workers;
    cudaError_t err[spb_ctx::XFER_WORKERS];
    auto work = [&](int w) {
        cudaError_t e = cudaSetDevice(c->device);
        int b = 0;
        size_t pending_chunk[2] = {(size_t)-1, (size_t)-1};   // downloads: chunk whose DMA into buffer b is in flight
        for (size_t k = w; k < chunks.size() && e == cudaSuccess; k += (size_t)NW, b ^= 1) {
            const Chunk &ch = chunks[k];
            if (to_device) {
                e = cudaEventSynchronize(c->xfer_ev[w][b]);                       // the buffer's previous DMA has finished
                if (e != cudaSuccess) break;
                memcpy(c->xfer_buf[w][b], ch.host, ch.bytes);
                e = cudaMemcpyAsync(ch.dev, c->xfer_buf[w][b], ch.bytes, cudaMemcpyHostToDevice, c->xfer_stream[w]);
                if (e == cudaSuccess) e = cudaEventRecord(c->xfer_ev[w][b], c->xfer_stream[w]);
            } else {
                // start this chunk's DMA, then drain the other buffer (its DMA was started one round ago)
                e = cudaMemcpyAsync(c->xfer_buf[w][b], ch.dev, ch.bytes, cudaMemcpyDeviceToHost, c->xfer_stream[w]);
                if (e == cudaSuccess) e = cudaEventRecord(c->xfer_ev[w][b], c->xfer_stream[w]);
                pending_chunk[b] = k;
                const int o = b ^ 1;
                if (e == cudaSuccess && pending_chunk[o] != (size_t)-1) {
                    e = cudaEventSynchronize(c->xfer_ev[w][o]);
                    if (e == cudaSuccess) memcpy(chunks[pending_chunk[o]].host, c->xfer_buf[w][o], chunks[pending_chunk[o]].bytes);
                    pending_chunk[o] = (size_t)-1;
                }
            }
        }
        if (!to_device)
            for (int o = 0; o < 2 && e == cudaSuccess; ++o)
                if (pending_chunk[o] != (size_t)-1) {
                    e = cudaEventSynchronize(c->xfer_ev[w][o]);
                    if (e == cudaSuccess) memcpy(chunks[pending_chunk[o]].host, c->xfer_buf[w][o], chunks[pending_chunk[o]].bytes);
                }
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->xfer_stream[w]);
        err[w] = e;
    };
    // downloads: what is read was produced on the context's stream; uploads: the destination blocks may have been handed
    // back to the pool by work that is still running there
    CK(cudaStreamSynchronize(c->stream));
    std::thread th[spb_ctx::XFER_WORKERS];
    for (int w = 1; w < NW; ++w) th[w] = std::thread(work, w);
    work(0);
    for (int w = 1; w < NW; ++w) th[w].join();
    for (int w = 0; w < NW; ++w)
        if (err[w] != cudaSuccess) return spb_fail(SPB_ERR_CUDA, "host transfer failed: %s", cudaGetErrorString(err[w]));
    return 0;
}

// ==================================================================================================
extern "C" {

const char *spb_last_error(void) { return g_last_error.c_str(); }
int spb_version(void) { return 100; }

int spb_ctx_create(int device, void *cuda_stream, spb_ctx **out) {
    if (!out) return spb_fail(SPB_ERR_ARG, "spb_ctx_create: out is null");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return spb_fail(SPB_ERR_CUDA, "no CUDA device available (%s); spsparse_b200 has no CPU fallback",
                        cudaGetErrorString(e));
    if (device < 0 || device >= count) return spb_fail(SPB_ERR_ARG, "device %d out of range (%d devices)", device, count);
    CK(cudaSetDevice(device));
    struct Undo {  // a failing set-up step below must not leak the context or its stream
        spb_ctx *c;
        ~Undo() {
            if (!c) return;
            if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
            delete c;
        }
    } undo{new spb_ctx()};
    spb_ctx *c = undo.c;
    c->device = device;
    c->stream = nullptr;
    c->own_stream = (cuda_stream == nullptr);
    if (c->own_stream) CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    else c->stream = (cudaStream_t)cuda_stream;
    CK(cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device));
    CK(cudaFuncSetAttribute(k_radix_pass<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RS_SMEM_BYTES));
    CK(cudaFuncSetAttribute(k_radix_pass<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RS_SMEM_BYTES));
    CK(cudaFuncSetAttribute(k_reduce_segsort, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RfSmem)));
    CK(cudaFuncSetAttribute(k_radix_pass9<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)R9_SMEM_BYTES));
    CK(cudaFuncSetAttribute(k_radix_pass9<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)R9_SMEM_BYTES));
    CK(cudaFuncSetAttribute(k_radix_pass<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RS_SMEM_BYTES));
    CK(cudaFuncSetAttribute(k_radix_pass<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RS_SMEM_BYTES));
    CK(cudaFuncSetAttribute(k_radix_pass9<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)R9_SMEM_BYTES));
    CK(cudaFuncSetAttribute(k_radix_pass9<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)R9_SMEM_BYTES));
    c->bulk_load = getenv("SPB_BULK_LOAD") ? atoi(getenv("SPB_BULK_LOAD")) != 0 : true;
    const char *s = getenv("SPB_POOL_POISON");
    if (s) {  // one byte in hex: "00", "ff", "7f"
        char *end = nullptr;
        const unsigned long b = strtoul(s, &end, 16);
        if (!*s || *end || b > 0xff) return spb_fail(SPB_ERR_ARG, "SPB_POOL_POISON=%s: expected one byte in hex (00 .. ff)", s);
        c->pool.poison = (int)b;
        c->pool.stream = c->stream;
    }
    s = getenv("SPB_MERGE_MAX_PRODUCTS");
    c->merge_max_products = s ? (u32)strtoul(s, nullptr, 10) : 1024u;
    s = getenv("SPB_ESC_CHUNK");
    c->esc_chunk = s ? strtoull(s, nullptr, 10) : (1ull << 27);
    c->launches = 0;
    c->xfer_ready = false;
    s = getenv("SPB_HASH_MIN_PRODUCTS");
    c->hash_min_products = s ? (strcmp(s, "off") == 0 ? ~0ull : strtoull(s, nullptr, 10)) : 512ull;
    s = getenv("SPB_HASH_VARIANT");
    c->hash_variant = s ? atoi(s) : 2;  // R-MAT scale 20, numeric pass: 1 x 1024 threads 82 ms, 2 x 512 72.9 ms, 4 x 256 70.3 ms
    CK(cudaFuncSetAttribute(k_hash_symbolic, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(HASH_MAX_COLS / 8)));
    CK(cudaFuncSetAttribute(k_hash_numeric<1024, 10240, 16384>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(HashSmem<1024, 10240, 16384>)));
    CK(cudaFuncSetAttribute(k_hash_numeric<512, 5120, 8192>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(HashSmem<512, 5120, 8192>)));
    CK(cudaFuncSetAttribute(k_hash_numeric<256, 2560, 4096>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(HashSmem<256, 2560, 4096>)));
    if (c->esc_chunk < 1) c->esc_chunk = 1;
    undo.c = nullptr;
    *out = c;
    return SPB_OK;
}

int spb_ctx_destroy(spb_ctx *ctx) {
    if (!ctx) return SPB_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->xfer_ready)
        for (int w = 0; w < ctx->xfer_workers; ++w) {
            cudaStreamDestroy(ctx->xfer_stream[w]);
            for (int b = 0; b < 2; ++b) { cudaFreeHost(ctx->xfer_buf[w][b]); cudaEventDestroy(ctx->xfer_ev[w][b]); }
        }
    ctx->pool.destroy();
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return SPB_OK;
}

int spb_ctx_sync(spb_ctx *ctx) {
    if (!ctx) return spb_fail(SPB_ERR_ARG, "null context");
    CK(cudaStreamSynchronize(ctx->stream));
    return SPB_OK;
}

int spb_ctx_trim(spb_ctx *ctx, uint64_t *released_bytes) {
    if (!ctx) return spb_fail(SPB_ERR_ARG, "null context");
    CK(cudaSetDevice(ctx->device));
    std::lock_guard<std::mutex> g(ctx->pool.mu_);
    if (released_bytes) *released_bytes = ctx->pool.cached_bytes;
    ctx->pool.trim_locked();
    return SPB_OK;
}

int spb_host_prefault(void *p, uint64_t bytes) {
    if (!p || !bytes) return SPB_OK;
    unsigned nt = std::thread::hardware_concurrency();
    if (nt > 16) nt = 16;
    if (bytes < (64ull << 20) || nt < 2) nt = 1;
    constexpr uint64_t PAGE = 4096;
    auto work = [=](unsigned t) {
        volatile char *c = static_cast<volatile char *>(p);
        const uint64_t a = bytes * t / nt, b = bytes * (t + 1) / nt;
        if (a < b) c[a] = 0;
        // page-aligned addresses inside [a, b): one write per page
        const uint64_t base = reinterpret_cast<uintptr_t>(p);
        for (uint64_t o = ((base + a + PAGE - 1) & ~(PAGE - 1)) - base; o < b; o += PAGE) c[o] = 0;
    };
    if (nt == 1) { work(0); return SPB_OK; }
    std::vector<std::thread> th;
    for (unsigned t = 1; t < nt; ++t) th.emplace_back(work, t);
    work(0);
    for (auto &x : th) x.join();
    return SPB_OK;
}

int spb_ctx_launch_count(const spb_ctx *ctx, uint64_t *launches) {
    if (!ctx || !launches) return spb_fail(SPB_ERR_ARG, "null argument");
    *launches = ctx->launches;
    return SPB_OK;
}

int spb_ctx_device(const spb_ctx *ctx, int *device, void **cuda_stream) {
    if (!ctx) return spb_fail(SPB_ERR_ARG, "null context");
    if (device) *device = ctx->device;
    if (cuda_stream) *cuda_stream = (void *)ctx->stream;
    return SPB_OK;
}

// ---- COO handles ---------------------------------------------------------------------------------
static int coo_new(spb_ctx *ctx, int rank, const u64 *shape, u64 n, bool allocate, spb_coo **out) {
    if (!ctx || !out || !shape) return spb_fail(SPB_ERR_ARG, "null argument");
    if (rank != 1 && rank != 2) return spb_fail(SPB_ERR_ARG, "rank must be 1 or 2 (got %d)", rank);
    for (int k = 0; k < rank; ++k)
        if (shape[k] > (1ull << 31)) return spb_fail(SPB_ERR_ARG, "extent %llu exceeds the int32 index range", (ull)shape[k]);
    if (n >= (1ull << 31)) return spb_fail(SPB_ERR_TOO_LARGE, "%llu entries: the reference's own cap is 2^31 (algorithm.hpp:419)", (ull)n);
    spb_coo *a = new spb_coo();
    a->rank = rank;
    a->shape[0] = shape[0];
    a->shape[1] = rank > 1 ? shape[1] : 1;
    a->n = n;
    a->idx[0] = a->idx[1] = nullptr;
    a->val = nullptr;
    a->sort_order[0] = -1;
    a->sort_order[1] = 0;
    a->owned = allocate;
    a->row_start = nullptr;
    a->row_id = nullptr;
    a->nrows = 0;
    a->rows_valid = false;
    a->dense_ptr = nullptr;
    a->dense_ptr_owned = true;
    a->range_ptr = nullptr;
    a->range_lo = a->range_hi = 0;
    a->max_row_len = 0;
    if (allocate) {
        size_t cnt = n ? n : 1;
        cudaError_t e = cudaSetDevice(ctx->device);
        for (int k = 0; k < rank && e == cudaSuccess; ++k) e = ctx->pool.alloc((void **)&a->idx[k], cnt * sizeof(i32));
        if (e == cudaSuccess) e = ctx->pool.alloc((void **)&a->val, cnt * sizeof(double));
        if (e != cudaSuccess) {  // give back what was obtained
            for (int k = 0; k < 2; ++k) ctx->pool.release(a->idx[k]);
            ctx->pool.release(a->val);
            delete a;
            return spb_fail(SPB_ERR_CUDA, "device allocation for %llu entries failed: %s", (ull)n, cudaGetErrorString(e));
        }
    }
    *out = a;
    return SPB_OK;
}

static void drop_row_cache(spb_ctx *ctx, spb_coo *a) {
    if (ctx) {
        ctx->pool.release(a->row_start);
        ctx->pool.release(a->row_id);
        if (a->dense_ptr_owned) ctx->pool.release(a->dense_ptr);
        ctx->pool.release(a->range_ptr);
    }
    a->row_start = nullptr; a->row_id = nullptr; a->dense_ptr = nullptr; a->range_ptr = nullptr;
    a->rows_valid = false; a->nrows = 0; a->max_row_len = 0;
}

static void set_order(spb_coo *a, const int *so) {
    a->sort_order[0] = -1;
    a->sort_order[1] = 0;
    if (so && so[0] >= 0) {
        a->sort_order[0] = so[0];
        a->sort_order[1] = a->rank > 1 ? so[1] : 0;
    }
}

int spb_coo_alloc(spb_ctx *ctx, int rank, const uint64_t *shape, uint64_t n, spb_coo **out) {
    return coo_new(ctx, rank, shape, n, true, out);
}

int spb_coo_upload(spb_ctx *ctx, int rank, const uint64_t *shape, const int32_t *const *idx, const double *val,
                   uint64_t n, const int *sort_order, spb_coo **out) {
    if (n && (!idx || !val)) return spb_fail(SPB_ERR_ARG, "null data pointer");
    CKR(coo_new(ctx, rank, shape, n, true, out));
    spb_coo *a = *out;
    set_order(a, sort_order);
    XferJob jobs[3];
    int nj = 0;
    for (int k = 0; k < rank && n; ++k) {
        if (!idx[k]) { spb_coo_free(ctx, a); *out = nullptr; return spb_fail(SPB_ERR_ARG, "null index pointer for dimension %d", k); }
        jobs[nj++] = {a->idx[k], const_cast<int32_t *>(idx[k]), (size_t)n * sizeof(i32)};
    }
    if (n) jobs[nj++] = {a->val, const_cast<double *>(val), (size_t)n * sizeof(double)};
    // (the uploaded arrays are used on ctx->stream afterwards: the copies are complete when this returns)
    const int rc = nj ? staged_copy(ctx, jobs, nj, true) : 0;  // host buffers are free to go when we return
    if (rc) {
        spb_coo_free(ctx, a);
        *out = nullptr;
        return rc;
    }
    return SPB_OK;
}

int spb_coo_wrap_device(spb_ctx *ctx, int rank, const uint64_t *shape, int32_t *const *d_idx, double *d_val,
                        uint64_t n, const int *sort_order, spb_coo **out) {
    if (n && (!d_idx || !d_val)) return spb_fail(SPB_ERR_ARG, "null device pointer");
    CKR(coo_new(ctx, rank, shape, n, false, out));
    spb_coo *a = *out;
    for (int k = 0; k < rank; ++k) a->idx[k] = d_idx ? d_idx[k] : nullptr;
    a->val = d_val;
    set_order(a, sort_order);
    return SPB_OK;
}

int spb_coo_info(const spb_coo *a, int *rank, uint64_t *shape, uint64_t *n, int *sort_order) {
    if (!a) return spb_fail(SPB_ERR_ARG, "null array");
    if (rank) *rank = a->rank;
    for (int k = 0; k < a->rank; ++k) {
        if (shape) shape[k] = a->shape[k];
        if (sort_order) sort_order[k] = a->sort_order[k];
    }
    if (n) *n = a->n;
    return SPB_OK;
}

int spb_coo_device_ptrs(const spb_coo *a, int32_t **d_idx, double **d_val) {
    if (!a) return spb_fail(SPB_ERR_ARG, "null array");
    for (int k = 0; k < a->rank; ++k) if (d_idx) d_idx[k] = a->idx[k];
    if (d_val) *d_val = a->val;
    return SPB_OK;
}

int spb_coo_set_sorted(spb_coo *a, const int *sort_order) {
    if (!a) return spb_fail(SPB_ERR_ARG, "null array");
    if (a->rows_valid || a->dense_ptr)
        return spb_fail(SPB_ERR_ARG, "spb_coo_set_sorted: the array's row structure is already in use");
    set_order(a, sort_order);
    return SPB_OK;
}

int spb_coo_download(spb_ctx *ctx, const spb_coo *a, int32_t *const *idx, double *val) {
    if (!ctx || !a) return spb_fail(SPB_ERR_ARG, "null argument");
    CK(cudaSetDevice(ctx->device));
    XferJob jobs[3];
    int nj = 0;
    if (a->n) {
        for (int k = 0; k < a->rank; ++k)
            if (idx && idx[k]) jobs[nj++] = {a->idx[k], idx[k], (size_t)a->n * sizeof(i32)};
        if (val) jobs[nj++] = {a->val, val, (size_t)a->n * sizeof(double)};
    }
    if (nj) return staged_copy(ctx, jobs, nj, false);
    CK(cudaStreamSynchronize(ctx->stream));
    return SPB_OK;
}

int spb_coo_free(spb_ctx *ctx, spb_coo *a) {
    if (!a) return SPB_OK;
    if (a->owned && ctx) {
        for (int k = 0; k < 2; ++k) if (a->idx[k]) ctx->pool.release(a->idx[k]);
        if (a->val) ctx->pool.release(a->val);
    }
    drop_row_cache(ctx, a);
    delete a;
    return SPB_OK;
}

}  // extern "C"

// ==================================================================================================
// sort + duplicate-reduce core, shared by consolidate and by multiply's operand preparation
// ==================================================================================================
struct SortJob {
    SortInput in;      // pass-0 source and drop rule
    int bits_hi;       // significant bits of the leading key part
    int policy;        // POLICY_*
};

// Runs the radix passes over packed keys already in (keysA, valsA) [n_ptr entries, upper bound n_cap];
// the sorted data ends up in *keys_sorted / *vals_sorted (one of the two buffer pairs).
template <typename InT, typename OutT>
static int exclusive_scan(spb_ctx *ctx, Scratch &ws, const InT *in, OutT *out, u64 n);

static int run_radix_passes(spb_ctx *ctx, Scratch &ws, int first_pass, int passes, u32 n_cap, const u32 *n_ptr,
                            u32 *hist, u64 *kA, double *vA, u64 *kB, double *vB, const SortInput *in0,
                            u64 **keys_sorted, double **vals_sorted, Timer *tm, int *mark_after_first, int shift0 = 0,
                            int digit_bits = RS_RADIX_BITS) {
    const u32 tiles = (u32)div_up(n_cap ? n_cap : 1, RS_TILE);
    const bool nine = digit_bits == R9_BITS;   // k_radix_pass9: 512 buckets per pass (hist and look-back rows are 512 wide)
    const u64 radix = nine ? R9_RADIX : RS_RADIX;
    u32 *lookback, *tickets;
    CKR(ws.zeroed(&lookback, (u64)passes * tiles * radix));
    CKR(ws.zeroed(&tickets, (u64)passes));
    u64 *kin = kA, *kout = kB;
    double *vin = vA, *vout = vB;
    for (int p = 0; p < passes; ++p) {
        PassArgs a;
        a.n_ptr = n_ptr;
        a.bucket_start = hist + (u64)p * radix;
        a.lookback = lookback + (u64)p * tiles * radix;
        a.ticket = tickets + p;
        a.shift = shift0 + p * digit_bits;
        a.rank_mode = getenv("SPB_RANK_MODE") ? atoi(getenv("SPB_RANK_MODE")) : 0;
        if (p == 0 && first_pass == 0) {
            // pass 0 reads the caller's arrays and writes buffer A
            a.keys_in = nullptr; a.vals_in = nullptr; a.keys_out = kA; a.vals_out = vA;
            // full tiles through the bulk-copy kernel when the caller's arrays allow 16-byte transfers, the last (partial)
            // tile -- or everything -- through the plain one; both draw tile numbers from the same ticket counter
            const bool aligned = ((((uintptr_t)in0->hi) | ((uintptr_t)in0->lo) | ((uintptr_t)in0->val)) & 15u) == 0;
            const u32 tiles_bulk = (ctx->bulk_load && aligned) ? n_cap / RS_TILE : 0;
            if (tiles_bulk) {
                ++ctx->launches;
                if (nine) k_radix_pass9<true, true><<<tiles_bulk, RS_THREADS, R9_SMEM_BYTES, ctx->stream>>>(a, *in0);
                else k_radix_pass<true, true><<<tiles_bulk, RS_THREADS, RS_SMEM_BYTES, ctx->stream>>>(a, *in0);
            }
            if (tiles > tiles_bulk) {
                ++ctx->launches;
                if (nine) k_radix_pass9<true><<<tiles - tiles_bulk, RS_THREADS, R9_SMEM_BYTES, ctx->stream>>>(a, *in0);
                else k_radix_pass<true><<<tiles - tiles_bulk, RS_THREADS, RS_SMEM_BYTES, ctx->stream>>>(a, *in0);
            }
            kin = kA; vin = vA; kout = kB; vout = vB;
            if (tm) *mark_after_first = tm->mark();
        } else {
            a.keys_in = kin; a.vals_in = vin; a.keys_out = kout; a.vals_out = vout;
            SortInput dummy;
            memset(&dummy, 0, sizeof dummy);
            ++ctx->launches;
            if (ctx->bulk_load) {
                if (nine) k_radix_pass9<false, true><<<tiles, RS_THREADS, R9_SMEM_BYTES, ctx->stream>>>(a, dummy);
                else k_radix_pass<false, true><<<tiles, RS_THREADS, RS_SMEM_BYTES, ctx->stream>>>(a, dummy);
            } else {
                if (nine) k_radix_pass9<false><<<tiles, RS_THREADS, R9_SMEM_BYTES, ctx->stream>>>(a, dummy);
                else k_radix_pass<false><<<tiles, RS_THREADS, RS_SMEM_BYTES, ctx->stream>>>(a, dummy);
            }
            u64 *tk = kin; kin = kout; kout = tk;
            double *tv = vin; vin = vout; vout = tv;
        }
    }
    CK(cudaGetLastError());
    *keys_sorted = kin;
    *vals_sorted = vin;
    return 0;
}

// Sorts job.in by (hi,lo), applies the drop rule and the duplicate policy, writes the result into
// out_hi/out_lo/out_val (capacity in.n each) and returns the counts.
static int sort_reduce(spb_ctx *ctx, const SortJob &job, i32 *out_hi, i32 *out_lo, double *out_val,
                       u32 *h_kept, u32 *h_out, spb_consolidate_stats *st, u32 *row_start = nullptr,
                       i32 *row_id = nullptr, u32 *h_rows = nullptr) {
    const SortInput &in = job.in;
    const u32 n = in.n;
    const int key_bits = job.bits_hi + in.bits_lo;
    int passes_full = (key_bits + RS_RADIX_BITS - 1) / RS_RADIX_BITS;
    if (passes_full < 1) passes_full = 1;
    if (passes_full > RS_MAX_PASSES) return spb_fail(SPB_ERR_ARG, "key of %d bits is too wide", key_bits);
    // Radix passes over the row part only + one in-row column sort (k_segment_sort) when that saves at least one pass
    int passes_row = (job.bits_hi + RS_RADIX_BITS - 1) / RS_RADIX_BITS;
    if (passes_row < 1) passes_row = 1;
    // ... and the rows are short: the in-row sort compares every entry with the rest of its row (config 5, 5 per row:
    // 36.3 -> 28.4 ms; config 2, 12 per row: 12.8 -> 10.8 ms).  The average over the POSSIBLE rows is what is known up
    // front; rows longer than SEG_MAX take the fallback inside the branch below.
    const char *seg_env = getenv("SPB_SEGMENT_SORT");  // "0" never, "1" whenever it saves a pass, unset: heuristic
    // (small arrays keep the plain passes: a saved pass is microseconds there, the extra read-back of the long-row count
    // and a possible fallback are not -- R-MAT scale 20's 4 M-entry operand went 0.85 -> 2.3 ms with it)
    const bool seg_short = (double)n <= 16.0 * (double)in.extent_hi && n >= (1u << 23);
    const char *walk_env = getenv("SPB_SEGMENT_WALK");
    const bool seg_walk = walk_env ? atoi(walk_env) != 0 : (double)n <= 6.0 * (double)in.extent_hi;  // very short rows: neighbour walk
    // SPB_SEGMENT_WALK=2: the walk on shuffles for rows of at most 5 entries (k_segment_sort_shfl) -- bit-identical, measured
    // slower than the shared-memory walk (22.4 against 21.1 ms on the config 5 block: 16 shuffles per 24 entries keep the SM's
    // one shuffle unit busy), so not the default
    const bool seg_shfl = walk_env && atoi(walk_env) == 2;
    const bool seg = in.bits_lo > 0 && passes_full - passes_row >= 2 &&
                     (seg_env ? atoi(seg_env) != 0 : seg_short);
    // 9-bit digits (k_radix_pass9) when they cover the same bits in fewer passes -- a 27-bit row part takes three
    // passes instead of four (SPB_RADIX9)
    const int cover_bits = seg ? job.bits_hi : key_bits;
    const char *r9_env = getenv("SPB_RADIX9");
    const int passes8 = seg ? passes_row : passes_full;
    const int passes9 = cover_bits > 0 ? (cover_bits + R9_BITS - 1) / R9_BITS : 1;
    // default: on where it was measured -- the row passes of a large array (the heuristic's own choice of the row-pass
    // organisation, which needs 2^23 entries); "1" = wherever it saves a pass, "0" = never
    const bool nine_wanted = r9_env ? atoi(r9_env) != 0 : (seg && !seg_env);
    const bool nine = nine_wanted && passes9 < passes8;
    const int digit_bits = nine ? R9_BITS : RS_RADIX_BITS;
    const int passes = nine ? passes9 : passes8;
    const int shift0 = seg ? in.bits_lo : 0;
    if (n >= (1u << 31)) return spb_fail(SPB_ERR_TOO_LARGE, "%u entries: one sort holds fewer than 2^31 (the reference's own cap, algorithm.hpp:419)", n);
    Scratch ws(ctx);
    Timer tm(ctx->stream);
    const int t0 = tm.mark();

    u32 *hist, *counters;  // counters: [0] kept, [1] out-of-bounds flag, [2] out count, [3] long runs
    u64 *first_kept;
    CKR(ws.zeroed(&hist, (u64)passes * (nine ? R9_RADIX : RS_RADIX)));
    CKR(ws.zeroed(&counters, 8));
    CKR(ws.get(&first_kept, 2));
    CK(cudaMemsetAsync(first_kept, 0xFF, 2 * sizeof(u64), ctx->stream));
    SortInput in0 = in;
    in0.first_kept = first_kept;
    const u32 sgrid = (u32)ctx->sm_count * 4;
    if (in.drop_nan) {
        ++ctx->launches, k_first_kept_key<<<grid_for(n, 256, sgrid * 2), 256, 0, ctx->stream>>>(in0, first_kept);
        ++ctx->launches, k_first_kept_pos<<<grid_for(n, 256, sgrid * 2), 256, 0, ctx->stream>>>(in0, first_kept);
    }
    // 128-bit loads when the caller's arrays allow them (SPB_VEC_LOAD=0: the scalar kernels)
    const bool vec4 = ((((uintptr_t)in0.hi) | ((uintptr_t)in0.lo) | ((uintptr_t)in0.val)) & 15u) == 0 && n >= 4096 &&
                      !(getenv("SPB_VEC_LOAD") && atoi(getenv("SPB_VEC_LOAD")) == 0);
    if (nine) {
        ++ctx->launches;
        if (vec4) k_sort_hist_v4<9><<<grid_for(n / 4, 512, sgrid), 512, 0, ctx->stream>>>(in0, passes, shift0, hist, counters);
        else k_sort_hist9<<<grid_for(n, 512, sgrid), 512, 0, ctx->stream>>>(in0, passes, shift0, hist, counters);
        ++ctx->launches, k_bucket_starts9<<<passes, R9_RADIX / 2, 0, ctx->stream>>>(hist);
    } else {
        ++ctx->launches;
        if (vec4) k_sort_hist_v4<8><<<grid_for(n / 4, 512, sgrid), 512, 0, ctx->stream>>>(in0, passes, shift0, hist, counters);
        else k_sort_hist<<<grid_for(n, 512, sgrid), 512, 0, ctx->stream>>>(in0, passes, shift0, hist, counters);
        ++ctx->launches, k_bucket_starts<<<passes, RS_RADIX, 0, ctx->stream>>>(hist);
    }
    CK(cudaGetLastError());

    u64 *kA, *kB = nullptr, *ks;
    double *vA, *vB = nullptr, *vs;
    CKR(ws.get(&kA, n));
    CKR(ws.get(&vA, n));
    if (passes > 1 || seg) { CKR(ws.get(&kB, n)); CKR(ws.get(&vB, n)); }
    int t_p0 = t0;
    CKR(run_radix_passes(ctx, ws, 0, passes, n, counters, hist, kA, vA, kB, vB, &in0, &ks, &vs, &tm, &t_p0, shift0, digit_bits));
    const int t_passes = tm.mark();
    // SPB_FUSED_REDUCE=1: the in-row column sort runs inside the reduce pass (k_reduce_segsort) instead of as a pass of
    // its own.  It has no path for rows longer than SEG_MAX: it counts their entries, and if there are any its output
    // is discarded and the separate kernels run after all (second trip of the loop below).
    const char *fused_env = getenv("SPB_FUSED_REDUCE");
    bool fused = seg && seg_walk && fused_env && atoi(fused_env) != 0;
    u32 h[6];
    int t1 = t_passes, t2 = t_passes;
    u64 *const ks_rows = ks;      // grouped by row, insertion order inside: what both variants start from
    double *const vs_rows = vs;
    // One host synchronisation per consolidate in the common case: the in-row sort and the reduce pass are both launched
    // before the counters are read.  Only when rows longer than SEG_MAX turn up (hub rows) is the reduce pass run again,
    // after those rows have been re-sorted by their full key.
    bool long_rows_fixed = false;
    // SPB_REDUCE_WARP (default 1): the reduce pass runs a warp per 256-entry tile (k_reduce_warp).  After an in-row sort the
    // tiles' places in the output come from the head counts that kernel produced (scanned here), not from a look-back;
    // "0": a block per 2048-entry tile with a look-back (k_reduce_by_key), "2": a warp per tile with a look-back everywhere.
    const int rw_mode = getenv("SPB_REDUCE_WARP") ? atoi(getenv("SPB_REDUCE_WARP")) : 1;
    const u32 wtiles = (u32)div_up(div_up(n ? n : 1, RW_TILE), RW_WARPS) * RW_WARPS;   // warp tiles, whole blocks
    for (int attempt = 0;; ++attempt) {
        ks = ks_rows; vs = vs_rows;
        u64 *ko = (ks == kA) ? kB : kA;
        double *vo = (vs == vA) ? vB : vA;
        const u32 stiles = (u32)div_up(n, SG_TILE);
        u64 *tile_off = nullptr;   // exclusive prefix of the reduce tiles' head counts, when the in-row sort counted them
        if (seg && !fused) {
            // rows are grouped (insertion order inside): order every row by column
            if (!long_rows_fixed) {
                u64 *tile_cnt = nullptr;
                if (rw_mode == 1) {
                    CKR(ws.zeroed(&tile_cnt, (u64)wtiles + 2));
                    CKR(ws.get(&tile_off, (u64)wtiles + 2));
                }
                const int keep_all = job.policy == POLICY_KEEP_ALL;
                ++ctx->launches;
                if (seg_shfl) k_segment_sort_shfl<<<stiles, SG_THREADS, 0, ctx->stream>>>(ks, vs, counters, in.bits_lo, ko, vo, nullptr, counters + 5, tile_cnt, keep_all);
                else if (seg_walk) k_segment_sort_walk<<<stiles, SG_THREADS, 0, ctx->stream>>>(ks, vs, counters, in.bits_lo, ko, vo, nullptr, counters + 5, tile_cnt, keep_all);
                else k_segment_sort<<<stiles, SG_THREADS, 0, ctx->stream>>>(ks, vs, counters, in.bits_lo, ko, vo, nullptr, counters + 5, tile_cnt, keep_all);
                CK(cudaGetLastError());
                if (tile_cnt) CKR((exclusive_scan<u64, u64>(ctx, ws, tile_cnt, tile_off, (u64)wtiles + 1)));
            } else {
                // rows longer than SEG_MAX exist (h[0] kept entries, h[5] of them in such rows): their entries (left in place
                // above) are pulled out in order, sorted by the full key with the radix passes, and put back -- the
                // pulled-out sequence is ascending in the row, so sorted position i goes back where gathered position i came from
                const u32 n_kept = h[0], h_long = h[5];
                unsigned char *flags;
                u64 *slot, *lk, *lk2, *lks;
                double *lv, *lv2, *lvs;
                u32 *lhist, *lcount;
                CKR(ws.get(&flags, n_kept));
                CKR(ws.get(&slot, (u64)n_kept + 1));
                CK(cudaMemsetAsync(counters + 5, 0, sizeof(u32), ctx->stream));
                ++ctx->launches;
                if (seg_shfl) k_segment_sort_shfl<<<stiles, SG_THREADS, 0, ctx->stream>>>(ks, vs, counters, in.bits_lo, ko, vo, flags, counters + 5);
                else if (seg_walk) k_segment_sort_walk<<<stiles, SG_THREADS, 0, ctx->stream>>>(ks, vs, counters, in.bits_lo, ko, vo, flags, counters + 5);
                else k_segment_sort<<<stiles, SG_THREADS, 0, ctx->stream>>>(ks, vs, counters, in.bits_lo, ko, vo, flags, counters + 5);
                CKR((exclusive_scan<unsigned char, u64>(ctx, ws, flags, slot, n_kept)));
                CKR(ws.get(&lk, h_long)); CKR(ws.get(&lv, h_long)); CKR(ws.get(&lk2, h_long)); CKR(ws.get(&lv2, h_long));
                CKR(ws.zeroed(&lhist, (u64)passes_full * RS_RADIX));
                CKR(ws.zeroed(&lcount, 8));
                CK(cudaMemcpyAsync(lcount, &h_long, sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
                ++ctx->launches, k_gather_flagged<<<grid_for(n_kept, 256, sgrid * 4), 256, 0, ctx->stream>>>(ks, vs, flags, slot, n_kept, lk, lv);
                ++ctx->launches, k_keys_hist<<<grid_for(h_long, 512, sgrid), 512, 0, ctx->stream>>>(lk, h_long, passes_full, lhist);
                ++ctx->launches, k_bucket_starts<<<passes_full, RS_RADIX, 0, ctx->stream>>>(lhist);
                CKR(run_radix_passes(ctx, ws, 1, passes_full, h_long, lcount, lhist, lk, lv, lk2, lv2, nullptr, &lks, &lvs, nullptr, nullptr));
                ++ctx->launches, k_scatter_flagged<<<grid_for(n_kept, 256, sgrid * 4), 256, 0, ctx->stream>>>(lks, lvs, flags, slot, n_kept, ko, vo);
                CK(cudaGetLastError());
            }
            ks = ko; vs = vo;
        }
        t1 = tm.mark();

        // the reduce pass
        const bool rwarp = !fused && (tile_off != nullptr || rw_mode == 2);
        const u32 rtiles = rwarp ? wtiles / RW_WARPS : (u32)div_up(n, RK_TILE);   // blocks
        ReduceArgs ra;
        memset(&ra, 0, sizeof ra);
        ra.keys = ks; ra.vals = vs; ra.n_ptr = counters; ra.bits_lo = in.bits_lo; ra.policy = job.policy;
        ra.out_hi = out_hi; ra.out_lo = out_lo; ra.out_val = out_val; ra.out_count = counters + 2;
        if (tile_off) ra.state = tile_off;
        else CKR(ws.zeroed(&ra.state, rwarp ? (u64)wtiles : (u64)rtiles));
        CKR(ws.zeroed(&ra.ticket, 1));
        ra.long_cap = n / RK_LONG_RUN + 1;
        CKR(ws.get(&ra.long_list, 2ull * ra.long_cap));
        ra.long_count = counters + 3;
        ra.row_start = row_start; ra.row_id = row_id; ra.row_count = counters + 4;
        if (fused) {
            ++ctx->launches, k_reduce_segsort<<<rtiles, RK_THREADS, sizeof(RfSmem), ctx->stream>>>(ra, counters + 5);
        } else {
            if (rwarp && tile_off) ++ctx->launches, k_reduce_warp<false><<<rtiles, RW_THREADS, 0, ctx->stream>>>(ra);
            else if (rwarp) ++ctx->launches, k_reduce_warp<true><<<rtiles, RW_THREADS, 0, ctx->stream>>>(ra);
            else ++ctx->launches, k_reduce_by_key<MODE_CONSOLIDATE><<<rtiles, RK_THREADS, 0, ctx->stream>>>(ra);
            if (job.policy == POLICY_ADD || job.policy == POLICY_REPLACE)
                ++ctx->launches, k_long_runs<<<(u32)ctx->sm_count * 4, 256, 0, ctx->stream>>>(ra);
        }
        CK(cudaGetLastError());
        t2 = tm.mark();

        CK(cudaMemcpyAsync(h, counters, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (h[5] && !h[1] && attempt == 0 && seg) {
            // rows longer than SEG_MAX: the reduce pass just run saw them unsorted -- do it again.  The fused kernel has no
            // path for them: start over from the row-grouped array with the separate kernels.
            fused = false;
            long_rows_fixed = true;
            CK(cudaMemsetAsync(counters + 2, 0, 3 * sizeof(u32), ctx->stream));  // out count, long runs, rows (h[5] is re-counted)
            continue;
        }
        break;
    }
    if (h[1]) return spb_fail(SPB_ERR_ARG, "Sparse index out of bounds (an index is negative or >= its extent)");
    *h_kept = h[0];
    *h_out = h[2];
    if (h_rows) *h_rows = h[4];
    if (st) {
        st->n_in = n; st->n_kept = h[0]; st->n_out = h[2];
        st->key_bits = key_bits; st->passes = passes; st->digit_bits = digit_bits;
        st->ms_sort = tm.ms(t0, t1); st->ms_reduce = tm.ms(t1, t2); st->ms_total = tm.ms(t0, t2);
        st->ms_pass = passes > 1 ? tm.ms(t_p0, t_passes) / (float)(passes - 1) : 0.f;
    }
    return 0;
}

// consolidate `in` into a fresh array sorted by `so`; `ref_so` is the order the reference would have
// used at this call site (decides which NaNs form the "leading run" when zero_nan).
// ext_lo / ext_val (rank 2 only): caller-owned device buffers of in->n entries that receive the second sort dimension's index
// vector and the values instead of pool memory (the row-partitioned multiply has its shard of B consolidated straight
// into the buffer its peers read).
static int consolidate_core(spb_ctx *ctx, const spb_coo *in, const int *so, const int *ref_so, int policy,
                            bool drop_zero, int zero_nan, spb_coo **out, spb_consolidate_stats *st,
                            i32 *ext_lo = nullptr, double *ext_val = nullptr) {
    if (in->n >= (1ull << 31)) return spb_fail(SPB_ERR_TOO_LARGE, "%llu entries: one array holds fewer than 2^31 (the reference's own cap, algorithm.hpp:419)", (ull)in->n);
    spb_coo *r = nullptr;
    if (ext_lo && ext_val && in->rank == 2) {
        CKR(coo_new(ctx, in->rank, in->shape, in->n, false, &r));
        r->owned = true;   // the leading index vector comes from the pool; releasing the two external pointers is a no-op
        if (ctx->pool.alloc((void **)&r->idx[so[0]], (in->n ? in->n : 1) * sizeof(i32)) != cudaSuccess) {
            delete r;
            return spb_fail(SPB_ERR_CUDA, "out of device memory");
        }
        r->idx[so[1]] = ext_lo;
        r->val = ext_val;
    } else {
        CKR(coo_new(ctx, in->rank, in->shape, in->n, true, &r));
    }
    set_order(r, so);
    if (st) memset(st, 0, sizeof *st);
    if (in->n == 0) { *out = r; return SPB_OK; }  // algorithm.hpp:263,318
    const int d0 = so[0], d1 = in->rank > 1 ? so[1] : -1;
    SortJob job;
    memset(&job, 0, sizeof job);
    job.in.hi = in->idx[d0];
    job.in.lo = d1 >= 0 ? in->idx[d1] : nullptr;
    job.in.val = in->val;
    job.in.n = (u32)in->n;
    job.in.bits_lo = d1 >= 0 ? bits_for(in->shape[d1]) : 0;
    job.in.extent_hi = (u32)(in->shape[d0] > 0xffffffffull ? 0xffffffffu : in->shape[d0]);
    job.in.extent_lo = d1 >= 0 ? (u32)in->shape[d1] : 1u;
    job.in.drop_zero = drop_zero ? 1 : 0;
    job.in.drop_nan = (drop_zero && zero_nan) ? 1 : 0;
    const int r0 = ref_so[0], r1 = in->rank > 1 ? ref_so[1] : -1;
    job.in.ref_hi = in->idx[r0];
    job.in.ref_lo = r1 >= 0 ? in->idx[r1] : nullptr;
    job.in.ref_bits_lo = r1 >= 0 ? bits_for(in->shape[r1]) : 0;
    job.bits_hi = bits_for(in->shape[d0]);
    job.policy = policy;
    u32 kept = 0, nout = 0, nrows = 0;
    if (in->rank == 2) {  // the reduce pass also emits the compressed row starts of its output
        const u64 cap = (in->n < in->shape[d0] ? in->n : in->shape[d0]) + 1;
        if (ctx->pool.alloc((void **)&r->row_start, cap * sizeof(u32)) != cudaSuccess ||
            ctx->pool.alloc((void **)&r->row_id, cap * sizeof(i32)) != cudaSuccess) {
            spb_coo_free(ctx, r);
            return spb_fail(SPB_ERR_CUDA, "out of device memory");
        }
    }
    int rc = sort_reduce(ctx, job, r->idx[d0], d1 >= 0 ? r->idx[d1] : nullptr, r->val, &kept, &nout, st,
                         r->row_start, r->row_id, &nrows);
    if (rc) { spb_coo_free(ctx, r); return rc; }
    r->n = nout;
    if (in->rank == 2) {
        r->nrows = nrows;
        r->rows_valid = true;
        if (nout == 0) { const u32 z = 0; cudaMemcpyAsync(r->row_start, &z, sizeof z, cudaMemcpyHostToDevice, ctx->stream); }
    }
    *out = r;
    return SPB_OK;
}

static int check_order(const spb_coo *a, const int *so, const char *what) {
    if (!so) return spb_fail(SPB_ERR_ARG, "%s: sort_order is null", what);
    for (int k = 0; k < a->rank; ++k)
        if (a->n && !a->idx[k]) return spb_fail(SPB_ERR_ARG, "%s: array is in compressed (pointer) form", what);
    bool seen[2] = {false, false};
    for (int k = 0; k < a->rank; ++k) {
        if (so[k] < 0 || so[k] >= a->rank || seen[so[k]])
            return spb_fail(SPB_ERR_ARG, "%s: sort_order is not a permutation of the dimensions", what);
        seen[so[k]] = true;
    }
    return 0;
}

// ---- row structure -------------------------------------------------------------------------------
struct RowIndex {   // compressed rows of a sorted array (scratch-owned)
    u32 *start;     // [nrows+1]
    i32 *id;        // [nrows]
    u32 nrows;
};

// Compressed rows of a sorted array, cached in the handle after the first request.
static int build_row_index(spb_ctx *ctx, const spb_coo *a_const, RowIndex *ri) {
    spb_coo *a = const_cast<spb_coo *>(a_const);  // lazy cache, as VectorCooArray::dim_beginnings does
    if (!a->rows_valid && a->n && !a->idx[a->sort_order[0]])
        return spb_fail(SPB_ERR_ARG, "array in compressed (pointer) form has no row list; use it as the B operand only");
    if (!a->rows_valid) {
        const u32 n = (u32)a->n;
        const i32 *hi = a->idx[a->sort_order[0]];
        Scratch ws(ctx);
        u32 *rs = nullptr;
        i32 *rid = nullptr;
        CK(ctx->pool.alloc((void **)&rs, ((u64)n + 1) * sizeof(u32)));
        if (ctx->pool.alloc((void **)&rid, ((u64)n + 1) * sizeof(i32)) != cudaSuccess) {
            ctx->pool.release(rs);
            return spb_fail(SPB_ERR_CUDA, "out of device memory (row list of %u entries)", n);
        }
        a->row_start = rs; a->row_id = rid;
        u32 *count, *ticket;
        u64 *state;
        const u32 tiles = (u32)div_up(n ? n : 1, RH_TILE);
        CKR(ws.zeroed(&count, 1));
        CKR(ws.zeroed(&ticket, 1));
        CKR(ws.zeroed(&state, tiles));
        if (n) ++ctx->launches, k_row_heads<<<tiles, RH_THREADS, 0, ctx->stream>>>(hi, n, a->row_start, a->row_id, count, state, ticket);
        ++ctx->launches, k_row_sentinel<<<1, 1, 0, ctx->stream>>>(a->row_start, count, n);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(&a->nrows, count, sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        a->rows_valid = true;
    }
    ri->start = a->row_start;
    ri->id = a->row_id;
    ri->nrows = a->nrows;
    return 0;
}

template <typename InT, typename OutT>
static int exclusive_scan(spb_ctx *ctx, Scratch &ws, const InT *in, OutT *out, u64 n) {
    if (n == 0) { CK(cudaMemsetAsync(out, 0, sizeof(OutT), ctx->stream)); return 0; }
    const u32 tiles = (u32)div_up(n, SC_TILE);
    u64 *state;
    u32 *ticket;
    CKR(ws.zeroed(&state, tiles));
    CKR(ws.zeroed(&ticket, 1));
    ++ctx->launches, k_exclusive_scan<InT, OutT><<<tiles, SC_THREADS, 0, ctx->stream>>>(in, out, n, state, ticket);
    CK(cudaGetLastError());
    return 0;
}

// dense pointer over the `extent` values of the leading index of a sorted array (cached in the handle)
static int build_dense_ptr(spb_ctx *ctx, const spb_coo *a_const, u64 extent, u32 **ptr_out) {
    spb_coo *a = const_cast<spb_coo *>(a_const);
    if (!a->dense_ptr) {
        RowIndex ri;
        CKR(build_row_index(ctx, a, &ri));
        CK(ctx->pool.alloc((void **)&a->dense_ptr, (extent + 2) * sizeof(u32)));
        // straight from the compressed rows (one read, one write; nothing is read back: no host synchronisation)
        Scratch ws(ctx);
        DpGap *gaps = nullptr;
        u32 *n_gaps = nullptr;
        if (ri.nrows && extent + 1 - ri.nrows >= DP_LONG_GAP) {   // long stretches of empty rows are possible: list them
            CKR(ws.get(&gaps, (extent + 1) / DP_LONG_GAP + 1));
            CKR(ws.zeroed(&n_gaps, 1));
        }
        ++ctx->launches;
        if (ri.nrows) k_dense_ptr_from_rows<<<grid_for(ri.nrows, 256, (u32)ctx->sm_count * 16), 256, 0, ctx->stream>>>(ri.start, ri.id, ri.nrows, (u32)a->n, extent, a->dense_ptr, gaps, n_gaps);
        else k_fill_u32<<<grid_for(extent + 1, 256, (u32)ctx->sm_count * 16), 256, 0, ctx->stream>>>(a->dense_ptr, extent + 1, 0u);
        if (gaps) ++ctx->launches, k_fill_gaps<<<(u32)ctx->sm_count * 8, 256, 0, ctx->stream>>>(gaps, n_gaps, a->dense_ptr);
        CK(cudaGetLastError());
    }
    *ptr_out = a->dense_ptr;
    return 0;
}

// `bad` (device, zeroed by the caller): set when the vector's indices are not strictly ascending; the caller reads it
// back with its next synchronisation and fails the call (bad_scale_vector)
static int densify(spb_ctx *ctx, Scratch &ws, const spb_coo *v, u64 dim, double **dense, unsigned char **mask, u32 *bad) {
    CKR(ws.zeroed(dense, dim));
    if (mask) CKR(ws.zeroed(mask, dim));
    if (v->n) ++ctx->launches, k_densify<<<grid_for(v->n, 256, 1u << 16), 256, 0, ctx->stream>>>(v->idx[0], v->val, v->n, dim, *dense, mask ? *mask : nullptr, bad);
    CK(cudaGetLastError());
    return 0;
}
static int bad_scale_vector() {
    return spb_fail(SPB_ERR_ARG, "a scale vector (or a vector operand flagged sorted) is not strictly ascending in its index: the "
                    "reference joins these as sorted lists without repeats (xiter.hpp:146, 201)");
}

// ==================================================================================================
// multiply core on prepared operands
// ==================================================================================================
static int esc_sort_reduce(spb_ctx *ctx, u64 *kA, double *vA, u32 count, int key_bits, int kbits,
                           const MMOperands &m, u32 row_lo, i32 *t_row, i32 *t_k, double *t_v, u32 *h_out) {
    Scratch ws(ctx);  // everything allocated here dies with this call
    int passes = (key_bits + RS_RADIX_BITS - 1) / RS_RADIX_BITS;
    if (passes < 1) passes = 1;
    u32 *hist, *counters;
    CKR(ws.zeroed(&hist, (u64)passes * RS_RADIX));
    CKR(ws.zeroed(&counters, 8));
    CK(cudaMemcpyAsync(counters, &count, sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    ++ctx->launches, k_keys_hist<<<grid_for(count, 512, (u32)ctx->sm_count * 4), 512, 0, ctx->stream>>>(kA, count, passes, hist);
    ++ctx->launches, k_bucket_starts<<<passes, RS_RADIX, 0, ctx->stream>>>(hist);
    u64 *kB, *ks;
    double *vB, *vs;
    CKR(ws.get(&kB, count));
    CKR(ws.get(&vB, count));
    // input is in A; passes ping-pong A->B->A...
    {
        const u32 tiles = (u32)div_up(count, RS_TILE);
        u32 *lookback, *tickets;
        CKR(ws.zeroed(&lookback, (u64)passes * tiles * RS_RADIX));
        CKR(ws.zeroed(&tickets, (u64)passes));
        u64 *kin = kA, *kout = kB;
        double *vin = vA, *vout = vB;
        SortInput dummy;
        memset(&dummy, 0, sizeof dummy);
        for (int p = 0; p < passes; ++p) {
            PassArgs a;
            a.keys_in = kin; a.vals_in = vin; a.keys_out = kout; a.vals_out = vout;
            a.n_ptr = counters;
            a.bucket_start = hist + (u64)p * RS_RADIX;
            a.lookback = lookback + (u64)p * tiles * RS_RADIX;
            a.ticket = tickets + p;
            a.shift = p * RS_RADIX_BITS;
            a.rank_mode = 0;
        a.rank_mode = getenv("SPB_RANK_MODE") ? atoi(getenv("SPB_RANK_MODE")) : 0;
            ++ctx->launches;
            if (ctx->bulk_load) k_radix_pass<false, true><<<tiles, RS_THREADS, RS_SMEM_BYTES, ctx->stream>>>(a, dummy);
            else k_radix_pass<false><<<tiles, RS_THREADS, RS_SMEM_BYTES, ctx->stream>>>(a, dummy);
            u64 *tk = kin; kin = kout; kout = tk;
            double *tv = vin; vin = vout; vout = tv;
        }
        ks = kin; vs = vin;
        CK(cudaGetLastError());
    }
    const u32 rtiles = (u32)div_up(count, RK_TILE);
    ReduceArgs ra;
    memset(&ra, 0, sizeof ra);
    ra.keys = ks; ra.vals = vs; ra.n_ptr = counters; ra.bits_lo = kbits; ra.policy = POLICY_ADD;
    ra.out_hi = t_row; ra.out_lo = t_k; ra.out_val = t_v; ra.out_count = counters + 2;
    CKR(ws.zeroed(&ra.state, rtiles));
    CKR(ws.zeroed(&ra.ticket, 1));
    ra.row_ids = m.arow_id; ra.row_base = (i32)row_lo; ra.si = m.si; ra.sk = m.sk; ra.C = m.C;
    ++ctx->launches, k_reduce_by_key<MODE_ESC><<<rtiles, RK_THREADS, 0, ctx->stream>>>(ra);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h_out, counters + 2, sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

struct EscChunk { i32 *row; i32 *k; double *v; u32 n; };

// Dynamic shared memory that a kernel does not use but that caps how many of its blocks share an SM.  The merge
// kernels are sensitive to it in both directions: more rows in flight hide the L2 latency of their dependent loads,
// but also spread L1/L2 over more partially written output sectors and more distinct B rows.
static size_t ballast_for_blocks(int blocks_per_sm, size_t static_smem) {
    if (blocks_per_sm <= 0) return 0;
    const size_t per = (size_t)(227 * 1024) / (size_t)blocks_per_sm;
    return per > static_smem + 1024 ? per - static_smem - 1024 : 0;
}
template <typename K> static int allow_ballast(K kernel) {
    static thread_local const void *done[16];
    static thread_local int n = 0;
    for (int i = 0; i < n; ++i) if (done[i] == (const void *)kernel) return 0;
    CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    if (n < 16) done[n++] = (const void *)kernel;
    return 0;
}

// A: consolidated, sorted by (a_row_dim, other).  B: consolidated, sorted by (b_inner_dim, other).
struct PreScale {   // scalej already in dense form (the row-partitioned multiply keeps it across steps and only rewrites the needed range)
    const double *sj;
    const unsigned char *sj_mask;
};

// What the numeric half of a multiply reads: everything the symbolic half found, all of it depending only on the pattern of
// the operands and the scale vectors (the register-merge count and the hash bin's bitmap pass read no values).  The device
// arrays belong to the Scratch the symbolic half was given.
struct MmState {
    MMOperands m;
    u64 nnz_a, nnz_b;
    ull h_stats[8];           // as multiply_core's stats[] (see k_esc_row_products)
    ull staged_blocks;
    int nl_fit, nl_num, local_carve, blk_num;
    bool local_count;
    unsigned char *row_cls;
    u32 *row_cnt;
    u64 *c_ptr;
    u64 nnz_c;                // counting outputs that will cancel to exactly 0
    HashArgs ha;
    u32 hash_cap;
    u32 h_items;
    bool items_ready;         // the hash bin's work items and window searches exist (mm_hash_items ran)
    std::vector<EscChunk> chunks;
    u32 *esc_first;
    int t_prep, t_mcount, t_bins, t_hcount, t_esc, t_sym;   // marks of the symbolic half; t_prep < 0: it ran on another timer
};

// The hash bin's work items (k_hash_items) and, for rows cut into several items, where every item's window begins in every B
// row (k_hash_splits): structure only, written into s.ha.
static int mm_hash_items(spb_ctx *ctx, Scratch &ws, MmState &s, Timer &tm, int *t_emit, int *t_split) {
    HashArgs &ha = s.ha;
    const MMOperands &m = s.m;
    const u32 cap = (u32)ctx->sm_count * 32;
    const u64 max_items = s.h_stats[5] + s.nnz_c / s.hash_cap + 1;
    CKR(ws.get(&ha.items, max_items));
    CKR(ws.get(&ha.item_key, max_items));
    ha.c_ptr = s.c_ptr;
    ++ctx->launches, k_hash_items<<<grid_for((u64)ha.nrows * 32, 256, (u32)ctx->sm_count * 8), 256, 0, ctx->stream>>>(m, ha);
    CK(cudaGetLastError());
    ull h_split = 0;
    *t_emit = *t_split = tm.mark();
    CK(cudaMemcpyAsync(&s.h_items, ha.n_items, sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&h_split, ha.split_total, sizeof(ull), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (h_split) {
        // rows cut into several items: where every item's column window begins in every B row of the row
        u32 *split;
        CKR(ws.get(&split, h_split));
        ++ctx->launches, k_hash_splits<<<s.h_items < cap * 4 ? s.h_items : cap * 4, 256, 0, ctx->stream>>>(m, ha, s.h_items, split);
        CK(cudaGetLastError());
        ha.split = split;
        *t_split = tm.mark();
    }
    s.items_ready = true;
    return 0;
}

// Symbolic half: prepares the operands (row index of A, dense pointer of B, densified scale vectors), bins the rows and places
// them.  *done: the call is complete without the numeric half (symbolic_only, or the one-pass merge went through and wrote
// `out`).  pattern (spb_mm_pattern_create): every row the register merge does not take goes to the hash bin -- expand-sort-
// compress forms values in its symbolic phase -- and the one-pass merge is never tried.
static int mm_symbolic(spb_ctx *ctx, Scratch &ws, double C, const spb_coo *si, const spb_coo *A, int a_row_dim,
                       const spb_coo *sj, const spb_coo *B, int b_inner_dim, const spb_coo *sk,
                       spb_coo *out, spb_mm_stats *st, Timer &tm, int t_begin, bool symbolic_only,
                       const PreScale *pre, bool pattern, MmState &s, bool *done) {
    *done = false;
    const int a_in = 1 - a_row_dim, b_col = 1 - b_inner_dim;
    const u64 m_rows = A->shape[a_row_dim], n_inner = A->shape[a_in], n_cols = B->shape[b_col];
    MMOperands m;
    memset(&m, 0, sizeof m);
    m.C = C;
    m.debug = getenv("SPB_MERGE_DEBUG") ? atoi(getenv("SPB_MERGE_DEBUG")) : 0;
    m.a_j = A->idx[a_in]; m.a_val = A->val; m.nnz_a = (u32)A->n;
    RowIndex ri;
    CKR(build_row_index(ctx, A, &ri));
    m.arow_id = ri.id; m.arow_start = ri.start; m.nrows = ri.nrows;
    u32 *bptr;
    CKR(build_dense_ptr(ctx, B, n_inner, &bptr));
    m.bptr = bptr; m.b_k = B->idx[b_col]; m.b_val = B->val;
    double *d;
    unsigned char *mask;
    u32 *bad_vec;
    CKR(ws.zeroed(&bad_vec, 1));
    if (si) { CKR(densify(ctx, ws, si, m_rows, &d, nullptr, bad_vec)); m.si = d; }
    if (pre) { m.sj = pre->sj; m.sj_mask = pre->sj_mask; }
    else if (sj) { CKR(densify(ctx, ws, sj, n_inner, &d, &mask, bad_vec)); m.sj = d; m.sj_mask = mask; }
    if (sk) { CKR(densify(ctx, ws, sk, n_cols, &d, nullptr, bad_vec)); m.sk = d; }
    const int t_prep = tm.mark();
    double h0 = now_ms();
    if (tracing()) fprintf(stderr, "[spb] mm: prepare done (host), alloc so far %.2f ms\n", g_alloc_ms);

    // ---- symbolic: bin every row; short rows are counted exactly by the merge itself -----------------
    const u32 nrows = m.nrows;
    u32 *row_cnt;
    u64 *ent_off = nullptr, *esc_f = nullptr, *esc_off, *c_ptr;
    unsigned char *row_cls;
    ull *stats;  // [0] F merged rows, [1] rows merged, [2] rows long, [3] F ESC rows, [4] F HASH rows, [5] rows HASH
    CKR(ws.get(&row_cls, nrows));
    CKR(ws.zeroed(&row_cnt, (u64)nrows + 1));
    ull *mstats;  // the count kernel's striped counters (MC_STRIPES x 8), summed on the host
    CKR(ws.zeroed(&stats, 8));
    CKR(ws.zeroed(&mstats, (u64)MC_STRIPES * 8));
    const u32 cap = (u32)ctx->sm_count * 32;
    // ---- one pass for matrices of short rows (k_merge_onepass): no symbolic phase at all ------------------------------------------
    // Tried when rows of A and of B are short on average (their product bounds the outputs per row) and the longest row of A,
    // if known, is a merge row; C is allocated for 16 outputs per row.  Anything the kernel cannot take makes it fail fast and
    // the two-pass path below runs as if nothing had happened.  Measured on the banded config: 17.8 ms against 7.3 + 8.8 ms for
    // count + numeric -- with ~3000 warps in flight a finishing warp walks ~90 look-back rounds back to the nearest inclusive
    // prefix, longer than its merges took -- so OFF unless SPB_MERGE_ONEPASS=1 (profiles/r02_notes.md).
    {
        const double avg_a_len = nrows ? (double)m.nnz_a / (double)nrows : 0.0;
        const double avg_b = n_inner ? (double)B->n / (double)n_inner : 0.0;
        const u64 cap_out = (u64)nrows * 16;
        const bool want = !symbolic_only && !pattern && nrows && avg_a_len * avg_b <= 40.0 && (A->max_row_len == 0 || A->max_row_len <= (u32)MERGE_MAX_LISTS) &&
                          cap_out < (1ull << 31) && cap_out * 16 <= (48ull << 30) &&
                          getenv("SPB_MERGE_ONEPASS") && atoi(getenv("SPB_MERGE_ONEPASS")) != 0;
        if (want) {
            spb_coo *Am1 = const_cast<spb_coo *>(A);
            if (!Am1->max_row_len) {   // picks the kernel build (registers per thread follow the longest row)
                u32 *mx;
                CKR(ws.zeroed(&mx, 1));
                ++ctx->launches, k_row_maxlen<<<grid_for(nrows, 256, cap), 256, 0, ctx->stream>>>(m.arow_start, nrows, mx);
                CK(cudaMemcpyAsync(&Am1->max_row_len, mx, sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
                CK(cudaStreamSynchronize(ctx->stream));
            }
            const u32 ml = A->max_row_len;
            if (ml <= (u32)MERGE_MAX_LISTS) {
                const u32 g = (u32)div_up(nrows, MR_THREADS);
                u64 *state;
                u32 *tk;
                ull *o1;
                i32 *ci = nullptr, *ck = nullptr;
                double *cv = nullptr;
                CKR(ws.zeroed(&state, (u64)g * (MR_THREADS / 32)));
                CKR(ws.zeroed(&tk, 2));
                CKR(ws.zeroed(&o1, 8 + (u64)MC_STRIPES * 8));
                if (ctx->pool.alloc((void **)&ci, cap_out * sizeof(i32)) != cudaSuccess || ctx->pool.alloc((void **)&ck, cap_out * sizeof(i32)) != cudaSuccess ||
                    ctx->pool.alloc((void **)&cv, cap_out * sizeof(double)) != cudaSuccess) {
                    cudaGetLastError();
                    ctx->pool.release(ci); ctx->pool.release(ck); ctx->pool.release(cv);
                } else {
                    ++ctx->launches;
                    if (ml <= 2) k_merge_onepass<2><<<g, MR_THREADS, 0, ctx->stream>>>(m, ctx->merge_max_products, state, tk, tk + 1, o1, ci, ck, cv);
                    else if (ml <= 4) k_merge_onepass<4><<<g, MR_THREADS, 0, ctx->stream>>>(m, ctx->merge_max_products, state, tk, tk + 1, o1, ci, ck, cv);
                    else if (ml <= 6) k_merge_onepass<6><<<g, MR_THREADS, 0, ctx->stream>>>(m, ctx->merge_max_products, state, tk, tk + 1, o1, ci, ck, cv);
                    else k_merge_onepass<8><<<g, MR_THREADS, 0, ctx->stream>>>(m, ctx->merge_max_products, state, tk, tk + 1, o1, ci, ck, cv);
                    CK(cudaGetLastError());
                    const int t_one = tm.mark();
                    ull h_o[8 + MC_STRIPES * 8];
                    u32 h_tk[2], h_badv = 0;
                    CK(cudaMemcpyAsync(h_o, o1, sizeof h_o, cudaMemcpyDeviceToHost, ctx->stream));
                    CK(cudaMemcpyAsync(h_tk, tk, sizeof h_tk, cudaMemcpyDeviceToHost, ctx->stream));
                    CK(cudaMemcpyAsync(&h_badv, bad_vec, sizeof h_badv, cudaMemcpyDeviceToHost, ctx->stream));
                    CK(cudaStreamSynchronize(ctx->stream));
                    if (h_badv) { ctx->pool.release(ci); ctx->pool.release(ck); ctx->pool.release(cv); return bad_scale_vector(); }
                    if (!h_tk[1]) {   // it went through
                        ull F1 = 0, rows1 = 0;
                        for (int sx = 0; sx < MC_STRIPES; ++sx) { F1 += h_o[8 + sx * 8]; rows1 += h_o[8 + sx * 8 + 1]; }
                        out->idx[0] = ci; out->idx[1] = ck; out->val = cv;
                        out->owned = true;
                        out->n = h_o[0];
                        if (st) {
                            st->products = F1; st->rows_merge = rows1; st->nnz_a = A->n; st->nnz_b = B->n; st->rows_a = nrows; st->nnz_c = h_o[0];
                            st->ms_prepare = tm.ms(t_begin, t_prep);
                            st->ms_symbolic = 0.f;
                            st->ms_numeric = tm.ms(t_prep, t_one);
                            st->ms_merge_numeric = st->ms_numeric;
                            st->ms_total = tm.ms(t_begin, t_one);
                        }
                        *done = true;
                        return SPB_OK;
                    }
                    ctx->pool.release(ci); ctx->pool.release(ck); ctx->pool.release(cv);
                }
            }
        }
    }

    // longest row of op(A): picks the leanest register-merge kernels that still cover every mergeable row.  Only the count
    // kernel's choice for long B rows needs it up front; otherwise the count kernel itself reports it (stats[6]) and it is
    // read back with the other counters -- one host round trip less per multiply of a freshly consolidated A.
    const double avg_b_len = n_inner ? (double)B->n / (double)n_inner : 0.0;
    spb_coo *Am = const_cast<spb_coo *>(A);
    const bool maxlen_up_front = !Am->max_row_len && nrows && (avg_b_len > 16.0 || getenv("SPB_MERGE_NL_COUNT"));
    if (maxlen_up_front) {
        u32 *mx;
        CKR(ws.zeroed(&mx, 1));
        ++ctx->launches, k_row_maxlen<<<grid_for(nrows, 256, cap), 256, 0, ctx->stream>>>(m.arow_start, nrows, mx);
        CK(cudaMemcpyAsync(&Am->max_row_len, mx, sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    const bool maxlen_known = A->max_row_len != 0;
    u32 a_maxlen = maxlen_known ? A->max_row_len : 0xffffffffu;   // unknown: the 8-list count kernel covers every row
    int nl_fit = a_maxlen <= 2 ? 2 : a_maxlen <= 4 ? 4 : a_maxlen <= 6 ? 6 : 8;
    // Measured (tools/merge_sweep.py): the lean builds win where B rows are long (config 3: count 2.92 -> 2.35 ms);
    // with 5-entry B rows (config 5) the count kernel is fastest as the 8-list build (7.0 ms against 9.8 ms for the
    // 6-list one at a third more warps), while the numeric kernel still prefers the lean one (10.9 -> 8.8 ms).
    const int nl_count = getenv("SPB_MERGE_NL_COUNT") ? atoi(getenv("SPB_MERGE_NL_COUNT")) : (avg_b_len > 16.0 ? nl_fit : 8);
    int nl_num = getenv("SPB_MERGE_NL_NUMERIC") ? atoi(getenv("SPB_MERGE_NL_NUMERIC")) : nl_fit;
    // (measured slower than the global merge on the banded config -- count 7.3 -> 11.0 ms, numeric 8.9 -> 16.3 ms: the staging
    // puts three barriers and four serialised round trips in front of every block -- so off unless SPB_MERGE_LOCAL=1;
    // profiles/r02_notes.md)
    const bool local_count = avg_b_len <= 16.0 && getenv("SPB_MERGE_LOCAL") && atoi(getenv("SPB_MERGE_LOCAL")) != 0;
    const int local_carve = getenv("SPB_MERGE_LOCAL_CARVE") ? atoi(getenv("SPB_MERGE_LOCAL_CARVE")) : -1;
    const int blk_count = getenv("SPB_MERGE_BLOCKS_COUNT") ? atoi(getenv("SPB_MERGE_BLOCKS_COUNT")) : 0;
    const int blk_num = getenv("SPB_MERGE_BLOCKS_NUMERIC") ? atoi(getenv("SPB_MERGE_BLOCKS_NUMERIC")) : 0;
    {
        const u32 g = (u32)div_up(nrows ? nrows : 1, 128);
        const size_t bal = ballast_for_blocks(blk_count, 0);
        ++ctx->launches;
        // L1 / shared-memory split (profiles/r01_notes.md, merge sweep): long B rows are read sequentially by every
        // thread and want the larger L1; short ones keep the driver's default
        const double avg_b_row = n_inner ? (double)B->n / (double)n_inner : 0.0;
        const int carve_c = getenv("SPB_MERGE_CARVEOUT_COUNT") ? atoi(getenv("SPB_MERGE_CARVEOUT_COUNT")) : (avg_b_row > 16.0 ? 25 : -1);
        // SPB_MERGE_LOCAL=1, short B rows: the LOCAL kernels (a block stages the stretch of B its rows reference in shared
        // memory; blocks whose rows reach too far fall back to the global merge by themselves)
#define SPB_LAUNCH_COUNT(NL) do { if (local_count) { \
            if (local_carve >= 0) CK(cudaFuncSetAttribute(k_merge_count<NL, true>, cudaFuncAttributePreferredSharedMemoryCarveout, local_carve)); \
            k_merge_count<NL, true><<<g, 128, 0, ctx->stream>>>(m, ctx->merge_max_products, row_cls, row_cnt, mstats); break; } \
        if (bal) CKR(allow_ballast(k_merge_count<NL>)); \
        if (carve_c >= 0) CK(cudaFuncSetAttribute(k_merge_count<NL>, cudaFuncAttributePreferredSharedMemoryCarveout, carve_c)); \
        k_merge_count<NL><<<g, 128, bal, ctx->stream>>>(m, ctx->merge_max_products, row_cls, row_cnt, mstats); } while (0)
        if (nl_count <= 2 && nl_fit <= 2) SPB_LAUNCH_COUNT(2);
        else if (nl_count <= 4 && nl_fit <= 4) SPB_LAUNCH_COUNT(4);
        else if (nl_count <= 6 && nl_fit <= 6) SPB_LAUNCH_COUNT(6);
        else SPB_LAUNCH_COUNT(8);
#undef SPB_LAUNCH_COUNT
    }
    CK(cudaGetLastError());
    const int t_mcount = tm.mark();
    ull h_stats[8];
    u32 *hash_rows = nullptr;
    u32 hash_small = 0;   // the first hash_small rows of hash_rows[] have at most HSM_CAP products
    u32 h_bad = 0;
    // the rows are placed right away, as if there were no long rows (true for banded / regridding matrices): the output
    // count then comes back with the counters in ONE round trip; with long rows the scan is repeated further down
    u64 nnz_c_spec = 0;
    CKR(ws.get(&c_ptr, (u64)nrows + 1));
    CKR((exclusive_scan<u32, u64>(ctx, ws, row_cnt, c_ptr, nrows)));
    ull h_mstats[MC_STRIPES * 8];
    CK(cudaMemcpyAsync(h_mstats, mstats, sizeof h_mstats, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&h_bad, bad_vec, sizeof h_bad, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&nnz_c_spec, c_ptr + nrows, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    memset(h_stats, 0, sizeof h_stats);
    ull staged_blocks = 0;   // LOCAL count kernel: blocks that ran from shared memory
    for (int sx = 0; sx < MC_STRIPES; ++sx) {
        staged_blocks += h_mstats[sx * 8 + 3];
        for (int q = 0; q < 3; ++q) h_stats[q] += h_mstats[sx * 8 + q];
        if (h_mstats[sx * 8 + 6] > h_stats[6]) h_stats[6] = h_mstats[sx * 8 + 6];
    }
    if (h_bad) return bad_scale_vector();
    if (!maxlen_known) {
        Am->max_row_len = (u32)h_stats[6];
        a_maxlen = A->max_row_len;
        nl_fit = a_maxlen <= 2 ? 2 : a_maxlen <= 4 ? 4 : a_maxlen <= 6 ? 6 : 8;
        if (!getenv("SPB_MERGE_NL_NUMERIC")) nl_num = nl_fit;
    }
    if (h_stats[2]) {
        // long rows exist: products per A entry, their prefix sums, products per long row
        u32 *ent_f;
        CKR(ws.get(&ent_f, m.nnz_a));
        CKR(ws.get(&ent_off, (u64)m.nnz_a + 1));
        CKR(ws.get(&esc_f, nrows));
        ++ctx->launches, k_entry_products<<<grid_for(m.nnz_a, 256, cap), 256, 0, ctx->stream>>>(m, A->idx[a_row_dim], ent_f);
        CKR((exclusive_scan<u32, u64>(ctx, ws, ent_f, ent_off, m.nnz_a)));
        // second-level bin: long rows with enough products use the bitmap + hash accumulators (needs the columns to fit the bitmap)
        const u64 hash_min = pattern ? 0 : ctx->hash_min_products;
        const bool hash_ok = hash_min != ~0ull;
        u32 *hash_rows_big = nullptr;
        if (hash_ok) { CKR(ws.get(&hash_rows, h_stats[2])); CKR(ws.get(&hash_rows_big, h_stats[2])); }
        // rows of at most HSM_CAP products: columns listed by a sort in shared memory (SPB_HASH_SMALL=0: everything by bitmap)
        // -- for matrices wider than the bitmap, where a row costs one bitmap unit PER COLUMN WINDOW (2^24 columns: 11): measured
        // 3.67 -> 2.69 s of config 4's sweep; with one window (R-MAT scale 20) the bitonic sort loses to the bitmap (29.8 -> 36.4 ms),
        // so there it needs SPB_HASH_SMALL=1
        const char *hs_env = getenv("SPB_HASH_SMALL");
        const bool wide = n_cols > (getenv("SPB_HASH_WIN_COLS") ? strtoull(getenv("SPB_HASH_WIN_COLS"), nullptr, 10) : (u64)HASH_MAX_COLS);
        const u64 small_max = (hs_env ? atoi(hs_env) != 0 : wide) ? (u64)HSM_CAP : 0;
        ++ctx->launches, k_esc_row_products<<<grid_for(nrows, 256, cap), 256, 0, ctx->stream>>>(m, ent_off, row_cls, esc_f, hash_min, small_max, hash_rows, hash_rows_big, stats);
        CK(cudaGetLastError());
        ull h_long[8];
        CK(cudaMemcpyAsync(h_long, stats, sizeof h_long, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        h_stats[3] = h_long[3]; h_stats[4] = h_long[4]; h_stats[5] = h_long[5];   // [0..2], [6] came from the count kernel's stripes
        hash_small = (u32)h_long[6];
        if (h_long[7])   // one list: the small rows, then the others
            CK(cudaMemcpyAsync(hash_rows + h_long[6], hash_rows_big, h_long[7] * sizeof(u32), cudaMemcpyDeviceToDevice, ctx->stream));
        ws.release(ent_f);
    }

    // ---- longer rows: bitmap count pass (the emit pass and the hash-accumulator numeric pass follow the placement) ----
    const int t_bins = tm.mark();
    HashArgs ha;
    memset(&ha, 0, sizeof ha);
    u32 hs_grid = 0;
    size_t hs_smem = 0;
    u32 hash_cap = ctx->hash_variant == 2 ? 2560u : ctx->hash_variant == 1 ? 5120u : 10240u;
    if (const char *e = getenv("SPB_HASH_ITEM_CAP")) {  // tests: cut rows into smaller work items
        const u32 v = (u32)strtoul(e, nullptr, 10);
        if (v >= 1 && v < hash_cap) hash_cap = v;
    }
    if (h_stats[5]) {
        ha.rows = hash_rows;
        ha.nrows = (u32)h_stats[5];
        // the bitmap covers win_cols columns; wider matrices are handled in column windows (SPB_HASH_WIN_COLS: tests)
        u64 win_cols = HASH_MAX_COLS;
        if (const char *e = getenv("SPB_HASH_WIN_COLS")) {
            const u64 v = strtoull(e, nullptr, 10) & ~31ull;
            if (v >= 32 && v < win_cols) win_cols = v;
        }
        ha.n_win = (u32)div_up(n_cols ? n_cols : 1, win_cols);
        ha.win_cols = (u32)win_cols;
        const u64 units = (u64)ha.nrows * ha.n_win;
        CKR(ws.zeroed(&ha.win_cnt, units));
        CKR(ws.get(&ha.win_pre, units));
        CKR(ws.get(&ha.seg_off, units));
        // the rows' output columns, written by the one bitmap pass before the rows are placed: at most one per product
        u64 tmp_cap = h_stats[4];
        if (tmp_cap > (u64)ha.nrows * n_cols) tmp_cap = (u64)ha.nrows * n_cols;
        CKR(ws.get(&ha.tmp_k, tmp_cap));
        ha.wpw = (u32)(div_up(div_up(ha.n_win > 1 ? win_cols : n_cols, 32), HS_WARPS) + 31) & ~31u;
        ha.cap = hash_cap;
        ha.no_sparse_walk = (getenv("SPB_HASH_SPARSE_WALK") && atoi(getenv("SPB_HASH_SPARSE_WALK")) == 0) ? 1u : 0u;
        ha.row_cnt = row_cnt;
        hs_grid = units < (u64)ctx->sm_count ? (u32)units : (u32)ctx->sm_count;
        hs_smem = (size_t)HS_WARPS * ha.wpw * sizeof(u32);
        CKR(ws.zeroed(&ha.next, 4));
        ha.shrunk = ha.next + 1;
        ha.n_items = ha.next + 2;
        CKR(ws.zeroed(&ha.split_total, 2));
        ha.tmp_cursor = ha.split_total + 1;
        CKR(ws.get(&ha.row_split, ha.nrows));
        ha.row0 = hash_small;
        if (ha.nrows > hash_small && ha.n_win > 1 && (u64)m.nnz_a * (ha.n_win - 1) <= (1ull << 30) && !getenv("SPB_HASH_NO_WIN_BOUNDS")) {
            // wide matrix: where every window begins in every B row, found by one parallel kernel (4 GB of positions at most;
            // beyond that the bitmap kernel searches for itself)
            u32 *wb;
            CKR(ws.get(&wb, (u64)m.nnz_a * (ha.n_win - 1)));
            ++ctx->launches, k_hash_win_bounds<<<ha.nrows < 65535u * 16u ? ha.nrows : 65535u * 16u, 128, 0, ctx->stream>>>(m, ha, wb);
            ha.win_bound = wb;
        }
        if (hash_small) ++ctx->launches, k_hash_symbolic_small<<<hash_small < (u32)ctx->sm_count * 6 ? hash_small : (u32)ctx->sm_count * 6, HSM_THREADS, 0, ctx->stream>>>(m, ha, hash_small);
        if (ha.nrows > hash_small) ++ctx->launches, k_hash_symbolic<<<hs_grid, HS_THREADS, hs_smem, ctx->stream>>>(m, ha);
        CK(cudaGetLastError());
    }

    // ---- long rows: expand-sort-compress into per-chunk temporaries -----------------------------
    const int t_hcount = tm.mark();
    std::vector<EscChunk> chunks;
    u64 esc_total = 0;
    u32 *esc_first = nullptr;
    if (h_stats[3]) {
        CKR(ws.get(&esc_off, (u64)nrows + 1));
        CKR((exclusive_scan<u64, u64>(ctx, ws, esc_f, esc_off, nrows)));
        CKR(ws.get(&esc_first, nrows));
        const u64 f_esc = h_stats[3];
        const u32 nchunks = (u32)div_up(f_esc, ctx->esc_chunk);
        u32 *rb;
        u64 *pb;
        CKR(ws.get(&rb, (u64)nchunks + 1));
        CKR(ws.get(&pb, (u64)nchunks + 1));
        ++ctx->launches, k_esc_chunks<<<(u32)div_up((u64)nchunks + 1, 128), 128, 0, ctx->stream>>>(esc_off, nrows, ctx->esc_chunk, nchunks, rb, pb);
        CK(cudaGetLastError());
        std::vector<u32> h_rb(nchunks + 1);
        std::vector<u64> h_pb(nchunks + 1);
        CK(cudaMemcpyAsync(h_rb.data(), rb, (nchunks + 1) * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(h_pb.data(), pb, (nchunks + 1) * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        const int kbits = bits_for(n_cols);
        for (u32 c = 0; c < nchunks; ++c) {
            const u32 r_lo = h_rb[c], r_hi = h_rb[c + 1];
            const u64 cnt64 = h_pb[c + 1] - h_pb[c];
            if (cnt64 == 0) continue;
            if (cnt64 >= (1ull << 31))
                return spb_fail(SPB_ERR_TOO_LARGE, "a single row of the product needs %llu intermediate products (>= 2^31)", (ull)cnt64);
            const u32 cnt = (u32)cnt64;
            const int key_bits = bits_for((u64)(r_hi - r_lo)) + kbits;
            u64 *kA;
            double *vA;
            i32 *t_row, *t_k;
            double *t_v;
            CKR(ws.get(&kA, cnt)); CKR(ws.get(&vA, cnt));
            CKR(ws.get(&t_row, cnt)); CKR(ws.get(&t_k, cnt)); CKR(ws.get(&t_v, cnt));
            ++ctx->launches, k_esc_expand<<<grid_for(cnt, 256, cap), 256, 0, ctx->stream>>>(m, esc_off, ent_off, r_lo, r_hi, h_pb[c], cnt, kbits, kA, vA);
            CK(cudaGetLastError());
            u32 nout = 0;
            CKR(esc_sort_reduce(ctx, kA, vA, cnt, key_bits, kbits, m, r_lo, t_row, t_k, t_v, &nout));
            ws.release(kA); ws.release(vA);
            esc_total += nout;
            if (esc_total >= (1ull << 31))
                return spb_fail(SPB_ERR_TOO_LARGE, "product has more than 2^31 entries; a VectorCooArray holds < 2^31 "
                                "(algorithm.hpp:419) -- multiply row panels of A instead");
            EscChunk ch;
            ch.n = nout;
            // shrink the temporaries to what was produced
            CKR(ws.get(&ch.row, nout)); CKR(ws.get(&ch.k, nout)); CKR(ws.get(&ch.v, nout));
            if (nout) {
                CK(cudaMemcpyAsync(ch.row, t_row, nout * sizeof(i32), cudaMemcpyDeviceToDevice, ctx->stream));
                CK(cudaMemcpyAsync(ch.k, t_k, nout * sizeof(i32), cudaMemcpyDeviceToDevice, ctx->stream));
                CK(cudaMemcpyAsync(ch.v, t_v, nout * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
                ++ctx->launches, k_esc_row_spans<<<grid_for(nout, 256, cap), 256, 0, ctx->stream>>>(ch.row, nout, esc_first, row_cnt);
                ++ctx->launches, k_esc_row_counts<<<grid_for(nout, 256, cap), 256, 0, ctx->stream>>>(ch.row, nout, esc_first, row_cnt);
            }
            ws.release(t_row); ws.release(t_k); ws.release(t_v);
            chunks.push_back(ch);
        }
        CK(cudaGetLastError());
    }

    // ---- place the rows ---------------------------------------------------------------------------
    const int t_esc = tm.mark();
    u64 nnz_c = nnz_c_spec;
    if (h_stats[2]) {   // long rows have filled in their counts since the speculative scan
        CKR((exclusive_scan<u32, u64>(ctx, ws, row_cnt, c_ptr, nrows)));
        CK(cudaMemcpyAsync(&nnz_c, c_ptr + nrows, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    const int t_sym = tm.mark();
    if (tracing()) fprintf(stderr, "[spb] mm: symbolic host %.2f ms, alloc total %.2f ms\n", now_ms() - h0, g_alloc_ms);
    if (symbolic_only) {
        // counts only (spb_mm_plan_symbolic): F and the bins are exact; nnz_c is exact except that outputs of the merge / hash bins whose
        // terms cancel to exactly 0 are still counted (the numeric pass is what finds them)
        if (st) {
            st->products = h_stats[0] + h_stats[3] + h_stats[4]; st->rows_merge = h_stats[1]; st->rows_esc = h_stats[2] - h_stats[5];
            st->products_esc = h_stats[3]; st->rows_hash = h_stats[5]; st->products_hash = h_stats[4];
            st->nnz_a = A->n; st->nnz_b = B->n; st->rows_a = nrows; st->nnz_c = nnz_c;
            st->ms_prepare = tm.ms(t_begin, t_prep);
            st->ms_symbolic = tm.ms(t_prep, t_sym);
            st->ms_total = tm.ms(t_begin, t_sym);
            st->ms_merge_count = tm.ms(t_prep, t_mcount);
            st->ms_hash_count = tm.ms(t_bins, t_hcount);
            st->ms_esc = tm.ms(t_hcount, t_esc);
        }
        *done = true;
        return SPB_OK;
    }
    s.m = m;
    s.nnz_a = A->n; s.nnz_b = B->n;
    memcpy(s.h_stats, h_stats, sizeof h_stats);
    s.staged_blocks = staged_blocks;
    s.nl_fit = nl_fit; s.nl_num = nl_num; s.local_carve = local_carve; s.blk_num = blk_num;
    s.local_count = local_count;
    s.row_cls = row_cls; s.row_cnt = row_cnt; s.c_ptr = c_ptr; s.nnz_c = nnz_c;
    s.ha = ha; s.hash_cap = hash_cap;
    s.h_items = 0; s.items_ready = false;
    s.chunks = chunks; s.esc_first = esc_first;
    s.t_prep = t_prep; s.t_mcount = t_mcount; s.t_bins = t_bins; s.t_hcount = t_hcount; s.t_esc = t_esc; s.t_sym = t_sym;
    return SPB_OK;
}

// Numeric half: forms C on the placement the symbolic half made, reading the values s.m.a_val / s.m.b_val.
static int mm_numeric(spb_ctx *ctx, Scratch &ws, MmState &s, spb_coo *out, spb_mm_stats *st, Timer &tm, int t_begin) {
    const MMOperands &m = s.m;
    const u32 nrows = m.nrows;
    const ull *h_stats = s.h_stats;
    u64 nnz_c = s.nnz_c;
    u64 *c_ptr = s.c_ptr;
    unsigned char *row_cls = s.row_cls;
    HashArgs &ha = s.ha;
    const u32 cap = (u32)ctx->sm_count * 32;
    const int blk_num = s.blk_num, local_carve = s.local_carve, nl_num = s.nl_num, nl_fit = s.nl_fit;
    const bool local_count = s.local_count;
    const ull staged_blocks = s.staged_blocks;
    const int t_sym = s.t_sym;
    const double h0 = now_ms();
    if (nnz_c >= (1ull << 31))
        return spb_fail(SPB_ERR_TOO_LARGE, "product has %llu entries; a VectorCooArray holds < 2^31 (algorithm.hpp:419) -- "
                        "form it in row panels (spb_mm_plan_create)", (ull)nnz_c);

    // ---- numeric ------------------------------------------------------------------------------------
    size_t cnt = nnz_c ? nnz_c : 1;
    CK(ctx->pool.alloc((void **)&out->idx[0], cnt * sizeof(i32)));
    CK(ctx->pool.alloc((void **)&out->idx[1], cnt * sizeof(i32)));
    CK(ctx->pool.alloc((void **)&out->val, cnt * sizeof(double)));
    out->owned = true;
    out->n = nnz_c;
    // register-merge rows: the (value-free) symbolic pass counted distinct columns; outputs whose sums turn out exactly 0 are
    // written as tombstones by the numeric pass and counted here; the compaction below closes the gaps (rare)
    u32 *mshrunk = nullptr;
    u32 h_mshrunk = 0;
    if (h_stats[1] && nnz_c)
        {
        CKR(ws.zeroed(&mshrunk, 1));
        ++ctx->launches;
        const u32 g = (u32)div_up(nrows, MR_THREADS);
        const int stage = getenv("SPB_MERGE_STAGE") ? atoi(getenv("SPB_MERGE_STAGE")) : 16;
        const size_t bal = ballast_for_blocks(blk_num, (size_t)MR_THREADS * 17 * 12);
        // numeric: the staging buffers (26 KB per block) compete with L1.  Rows with many products (long sequential
        // walks through B) ran best with 4 blocks and half of the array as L1, short rows with 7 blocks.
        const double avg_row_products = h_stats[1] ? (double)h_stats[0] / (double)h_stats[1] : 0.0;
        const int carve_n = getenv("SPB_MERGE_CARVEOUT_NUMERIC") ? atoi(getenv("SPB_MERGE_CARVEOUT_NUMERIC")) : (avg_row_products > 64.0 ? 50 : 75);
        // most blocks of the count kernel found their stretch of B small enough to stage: the numeric kernel stages too
        const bool local_num = local_count && stage == 16 && staged_blocks * 2 >= (ull)div_up(nrows, 128);
#define SPB_LAUNCH_NUM(NL, ST) do { if (local_num && ST == 16) { \
            if (local_carve >= 0) CK(cudaFuncSetAttribute(k_merge_numeric<NL, 16, true>, cudaFuncAttributePreferredSharedMemoryCarveout, local_carve)); \
            k_merge_numeric<NL, 16, true><<<g, MR_THREADS, 0, ctx->stream>>>(m, row_cls, c_ptr, out->idx[0], out->idx[1], out->val, mshrunk); break; } \
        if (bal) CKR(allow_ballast(k_merge_numeric<NL, ST>)); \
        if (carve_n >= 0) CK(cudaFuncSetAttribute(k_merge_numeric<NL, ST>, cudaFuncAttributePreferredSharedMemoryCarveout, carve_n)); \
        k_merge_numeric<NL, ST><<<g, MR_THREADS, bal, ctx->stream>>>(m, row_cls, c_ptr, out->idx[0], out->idx[1], out->val, mshrunk); } while (0)
        if (stage == 4) SPB_LAUNCH_NUM(8, 4);
        else if (stage == 8) SPB_LAUNCH_NUM(8, 8);
        else if (nl_num <= 2 && nl_fit <= 2) SPB_LAUNCH_NUM(2, 16);
        else if (nl_num <= 4 && nl_fit <= 4) SPB_LAUNCH_NUM(4, 16);
        else if (nl_num <= 6 && nl_fit <= 6) SPB_LAUNCH_NUM(6, 16);
        else SPB_LAUNCH_NUM(8, 16);
#undef SPB_LAUNCH_NUM
    }
    const int t_mnum = tm.mark();
    for (auto &ch : s.chunks)
        if (ch.n) ++ctx->launches, k_esc_copy<<<grid_for(ch.n, 256, cap), 256, 0, ctx->stream>>>(ch.row, ch.k, ch.v, ch.n, s.esc_first, c_ptr, m.arow_id, out->idx[0], out->idx[1], out->val);
    u32 h_shrunk = 0;
    int t_hemit0 = tm.mark(), t_hemit1 = t_hemit0, t_hsplit = t_hemit0, t_hnum = t_hemit0;
    if (h_stats[5] && nnz_c) {
        // the rows are placed: cut them into work items (the columns were listed by the bitmap pass of the symbolic phase)
        if (!s.items_ready) {
            CKR(mm_hash_items(ctx, ws, s, tm, &t_hemit1, &t_hsplit));
            t_hnum = t_hsplit;
        }
        ha.c_i = out->idx[0]; ha.c_k = out->idx[1]; ha.c_v = out->val;
        const u32 h_items = s.h_items;
        if (h_items) {
            ha.dbg = nullptr;
            if (tracing()) CKR(ws.zeroed(&ha.dbg, 16));
            ++ctx->launches;
            if (ctx->hash_variant == 2) {
                const u32 g = h_items < 4u * ctx->sm_count ? h_items : 4u * ctx->sm_count;
                k_hash_numeric<256, 2560, 4096><<<g, 256, sizeof(HashSmem<256, 2560, 4096>), ctx->stream>>>(m, ha, h_items);
            } else if (ctx->hash_variant == 1) {
                const u32 g = h_items < 2u * ctx->sm_count ? h_items : 2u * ctx->sm_count;
                k_hash_numeric<512, 5120, 8192><<<g, 512, sizeof(HashSmem<512, 5120, 8192>), ctx->stream>>>(m, ha, h_items);
            } else {
                const u32 g = h_items < (u32)ctx->sm_count ? h_items : (u32)ctx->sm_count;
                k_hash_numeric<1024, 10240, 16384><<<g, 1024, sizeof(HashSmem<1024, 10240, 16384>), ctx->stream>>>(m, ha, h_items);
            }
            CK(cudaGetLastError());
            t_hnum = tm.mark();
            CK(cudaMemcpyAsync(&h_shrunk, ha.shrunk, sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
            if (ha.dbg) {
                ull d[16];
                CK(cudaMemcpyAsync(d, ha.dbg, sizeof d, cudaMemcpyDeviceToHost, ctx->stream));
                CK(cudaStreamSynchronize(ctx->stream));
                fprintf(stderr, "[spb] mm hash numeric: %u items (%llu), %llu staged chunks, %llu steps (%llu warp-pipelined), %llu entry barriers\n", h_items, d[0], d[1], d[2], d[4], d[3]);
                const double tot = (double)(d[5] + d[6] + d[7] + d[8] + d[9]) / 100.0;
                fprintf(stderr, "[spb] mm hash numeric clocks: setup %.1f%%, staging %.1f%%, steps %.1f%%, warp-pipelined steps %.1f%%, output %.1f%%; %.0f clocks per item\n",
                        d[5] / tot, d[6] / tot, d[7] / tot, d[8] / tot, d[9] / tot, tot * 100.0 / (double)d[0]);
            }
        }
    }
    CK(cudaGetLastError());
    int t_num = tm.mark();   // (before the host looks at the tombstone counts: the wait is not kernel time)
    if (mshrunk) CK(cudaMemcpyAsync(&h_mshrunk, mshrunk, sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
    if (h_stats[5] || mshrunk) CK(cudaStreamSynchronize(ctx->stream));   // h_shrunk / h_mshrunk are in flight
    h_shrunk += h_mshrunk;
    if (h_shrunk) {
        // some outputs of the hash-accumulator or register-merge rows summed to exact zero and were dropped: close the gaps (rare)
        unsigned char *keep;
        u64 *slot;
        CKR(ws.get(&keep, nnz_c));
        CKR(ws.get(&slot, nnz_c + 1));
        ++ctx->launches, k_live_flags<<<grid_for(nnz_c, 256, cap), 256, 0, ctx->stream>>>(out->idx[0], nnz_c, keep);
        CKR((exclusive_scan<unsigned char, u64>(ctx, ws, keep, slot, nnz_c)));
        const u64 nnz2 = nnz_c - h_shrunk;
        i32 *i2, *k2;
        double *v2;
        size_t c2 = nnz2 ? nnz2 : 1;
        CK(ctx->pool.alloc((void **)&i2, c2 * sizeof(i32)));
        CK(ctx->pool.alloc((void **)&k2, c2 * sizeof(i32)));
        CK(ctx->pool.alloc((void **)&v2, c2 * sizeof(double)));
        ++ctx->launches, k_compact_entries<<<grid_for(nnz_c, 256, cap), 256, 0, ctx->stream>>>(nnz_c, keep, slot, out->idx[0], out->idx[1], out->val, i2, k2, v2);
        CK(cudaGetLastError());
        ctx->pool.release(out->idx[0]); ctx->pool.release(out->idx[1]); ctx->pool.release(out->val);
        out->idx[0] = i2; out->idx[1] = k2; out->val = v2;
        out->n = nnz_c = nnz2;
        t_num = tm.mark();
    }
    CK(cudaStreamSynchronize(ctx->stream));
    if (tracing()) fprintf(stderr, "[spb] mm: total host since prepare %.2f ms, alloc total %.2f ms\n", now_ms() - h0, g_alloc_ms);
    if (st) {
        st->products = h_stats[0] + h_stats[3] + h_stats[4]; st->rows_merge = h_stats[1]; st->rows_esc = h_stats[2] - h_stats[5];
        st->products_esc = h_stats[3]; st->rows_hash = h_stats[5]; st->products_hash = h_stats[4];
        st->nnz_a = s.nnz_a; st->nnz_b = s.nnz_b; st->rows_a = nrows; st->nnz_c = nnz_c;
        if (s.t_prep >= 0) {
            st->ms_prepare = tm.ms(t_begin, s.t_prep);
            st->ms_symbolic = tm.ms(s.t_prep, t_sym);
            st->ms_merge_count = tm.ms(s.t_prep, s.t_mcount);
            st->ms_hash_count = tm.ms(s.t_bins, s.t_hcount);
            st->ms_esc = tm.ms(s.t_hcount, s.t_esc);
        }
        st->ms_numeric = tm.ms(t_sym, t_num);
        st->ms_total = tm.ms(t_begin, t_num);
        st->ms_merge_numeric = tm.ms(t_sym, t_mnum);
        st->ms_hash_emit = tm.ms(t_hemit0, t_hemit1);
        st->ms_hash_splits = tm.ms(t_hemit1, t_hsplit);
        st->ms_hash_numeric = tm.ms(t_hsplit, t_hnum);
    }
    return SPB_OK;
}

static int multiply_core(spb_ctx *ctx, double C, const spb_coo *si, const spb_coo *A, int a_row_dim,
                         const spb_coo *sj, const spb_coo *B, int b_inner_dim, const spb_coo *sk,
                         spb_coo *out, spb_mm_stats *st, Timer &tm, int t_begin, bool symbolic_only = false,
                         const PreScale *pre = nullptr) {
    Scratch ws(ctx);
    MmState s;
    bool done = false;
    CKR(mm_symbolic(ctx, ws, C, si, A, a_row_dim, sj, B, b_inner_dim, sk, out, st, tm, t_begin, symbolic_only, pre, false, s, &done));
    if (done) return SPB_OK;
    return mm_numeric(ctx, ws, s, out, st, tm, t_begin);
}

// ==================================================================================================
extern "C" {

int spb_consolidate(spb_ctx *ctx, const spb_coo *in, const int *sort_order, int policy, int zero_nan,
                    spb_coo **out, spb_consolidate_stats *stats) {
    if (!ctx || !in || !out) return spb_fail(SPB_ERR_ARG, "spb_consolidate: null argument");
    CKR(check_order(in, sort_order, "spb_consolidate"));
    if (policy < 0 || policy > 2) return spb_fail(SPB_ERR_ARG, "unknown duplicate policy %d", policy);
    CK(cudaSetDevice(ctx->device));
    return consolidate_core(ctx, in, sort_order, sort_order, policy, true, zero_nan, out, stats);
}

int spb_coo_dense_ptr(spb_ctx *ctx, const spb_coo *a, uint32_t **d_ptr, uint64_t *extent) {
    if (!ctx || !a || !d_ptr) return spb_fail(SPB_ERR_ARG, "spb_coo_dense_ptr: null argument");
    if (a->rank != 2 || a->sort_order[0] < 0) return spb_fail(SPB_ERR_NOT_SORTED, "spb_coo_dense_ptr needs a consolidated rank-2 array");
    CK(cudaSetDevice(ctx->device));
    const u64 ext = a->shape[a->sort_order[0]];
    u32 *p = nullptr;
    CKR(build_dense_ptr(ctx, a, ext, &p));
    *d_ptr = p;
    if (extent) *extent = ext;
    return SPB_OK;
}

int spb_coo_dense_ptr_range(spb_ctx *ctx, const spb_coo *a_const, uint64_t lo, uint64_t hi, uint32_t **d_ptr) {
    if (!ctx || !a_const || !d_ptr) return spb_fail(SPB_ERR_ARG, "spb_coo_dense_ptr_range: null argument");
    spb_coo *a = const_cast<spb_coo *>(a_const);
    if (a->rank != 2 || a->sort_order[0] < 0) return spb_fail(SPB_ERR_NOT_SORTED, "spb_coo_dense_ptr_range needs a consolidated rank-2 array");
    if (lo > hi || hi > a->shape[a->sort_order[0]]) return spb_fail(SPB_ERR_ARG, "spb_coo_dense_ptr_range: bad range");
    if (!a->idx[a->sort_order[0]]) return spb_fail(SPB_ERR_ARG, "spb_coo_dense_ptr_range: compressed-form array");
    CK(cudaSetDevice(ctx->device));
    if (!a->range_ptr || a->range_lo != lo || a->range_hi != hi) {
        ctx->pool.release(a->range_ptr);
        a->range_ptr = nullptr;
        RowIndex ri;
        CKR(build_row_index(ctx, a, &ri));
        Scratch ws(ctx);
        const u64 span = hi - lo;
        u32 *len, *cnt;
        CKR(ws.zeroed(&len, span + 2));
        CKR(ws.get(&cnt, 1));
        CK(ctx->pool.alloc((void **)&a->range_ptr, (span + 3) * sizeof(u32)));
        CK(cudaMemcpyAsync(cnt, &ri.nrows, sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
        if (ri.nrows) ++ctx->launches, k_scatter_row_len_range<<<grid_for(ri.nrows, 256, 1u << 20), 256, 0, ctx->stream>>>(ri.start, ri.id, cnt, lo, hi, len);
        CKR((exclusive_scan<u32, u32>(ctx, ws, len, a->range_ptr, span + 1)));  // writes span + 2 values
        a->range_lo = lo; a->range_hi = hi;
    }
    *d_ptr = a->range_ptr + 1;
    return SPB_OK;
}

int spb_coo_wrap_csr(spb_ctx *ctx, const uint64_t *shape, int lead_dim, uint32_t *d_ptr, int32_t *d_other_idx,
                     double *d_val, uint64_t n, spb_coo **out) {
    if (!d_ptr || (n && (!d_other_idx || !d_val)) || (lead_dim | 1) != 1) return spb_fail(SPB_ERR_ARG, "spb_coo_wrap_csr: bad argument");
    CKR(coo_new(ctx, 2, shape, n, false, out));
    spb_coo *a = *out;
    a->idx[lead_dim] = nullptr;  // implicit in the pointer array
    a->idx[1 - lead_dim] = d_other_idx;
    a->val = d_val;
    a->sort_order[0] = lead_dim;
    a->sort_order[1] = 1 - lead_dim;
    a->dense_ptr = d_ptr;
    a->dense_ptr_owned = false;
    return SPB_OK;
}

int spb_sorted_permutation(spb_ctx *ctx, const spb_coo *in, const int *sort_order, uint64_t *perm) {
    if (!ctx || !in || (in->n && !perm)) return spb_fail(SPB_ERR_ARG, "spb_sorted_permutation: null argument");
    CKR(check_order(in, sort_order, "spb_sorted_permutation"));
    if (in->n == 0) return SPB_OK;
    CK(cudaSetDevice(ctx->device));
    // the radix sort moves a 64-bit payload with every key: give it the entry numbers
    Scratch ws(ctx);
    double *iota;
    CKR(ws.get(&iota, in->n));
    ++ctx->launches, k_iota_bits<<<grid_for(in->n, 256, 1u << 16), 256, 0, ctx->stream>>>(in->n, iota);
    CK(cudaGetLastError());
    spb_coo tmp = *in;
    tmp.val = iota;
    tmp.owned = false;
    spb_coo *sorted = nullptr;
    CKR(consolidate_core(ctx, &tmp, sort_order, sort_order, POLICY_KEEP_ALL, false, 0, &sorted, nullptr));
    int rc = SPB_OK;
    if (sorted->n != in->n) rc = spb_fail(SPB_ERR_CUDA, "sorted_permutation: lost entries (%llu of %llu)", (ull)sorted->n, (ull)in->n);
    if (!rc) {
        cudaError_t e = cudaMemcpyAsync(perm, sorted->val, in->n * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = spb_fail(SPB_ERR_CUDA, "sorted_permutation: %s", cudaGetErrorString(e));
    }
    spb_coo_free(ctx, sorted);
    return rc;
}

// ---- the steps either side of the path: copy / transpose / to_dense / to_sparse -------------------------------
int spb_coo_transpose(spb_ctx *ctx, const spb_coo *in, const int *perm, spb_coo **out) {
    if (!ctx || !in || !perm || !out) return spb_fail(SPB_ERR_ARG, "spb_coo_transpose: null argument");
    bool seen[2] = {false, false};
    for (int k = 0; k < in->rank; ++k) {
        if (perm[k] < 0 || perm[k] >= in->rank || seen[perm[k]]) return spb_fail(SPB_ERR_ARG, "spb_coo_transpose: not a permutation");
        seen[perm[k]] = true;
    }
    for (int k = 0; k < in->rank; ++k)
        if (in->n && !in->idx[k]) return spb_fail(SPB_ERR_ARG, "spb_coo_transpose: compressed-form array");
    CK(cudaSetDevice(ctx->device));
    uint64_t shape[2] = {1, 1};
    for (int k = 0; k < in->rank; ++k) shape[k] = in->shape[perm[k]];
    CKR(coo_new(ctx, in->rank, shape, in->n, true, out));
    spb_coo *r = *out;
    if (in->n) {
        for (int k = 0; k < in->rank; ++k)  // new dimension k takes old dimension perm[k]  (algorithm.hpp:51-54)
            CK(cudaMemcpyAsync(r->idx[k], in->idx[perm[k]], in->n * sizeof(i32), cudaMemcpyDeviceToDevice, ctx->stream));
        CK(cudaMemcpyAsync(r->val, in->val, in->n * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return SPB_OK;  // like a fresh VectorCooArray that was add()ed to: edit mode, not flagged sorted
}

int spb_coo_copy(spb_ctx *ctx, const spb_coo *in, spb_coo **out) {
    const int ident[2] = {0, 1};
    return spb_coo_transpose(ctx, in, ident, out);
}

int spb_coo_to_dense(spb_ctx *ctx, const spb_coo *in, int policy, double *dense) {
    if (!ctx || !in || !dense) return spb_fail(SPB_ERR_ARG, "spb_coo_to_dense: null argument");
    if (policy < 0 || policy > 2) return spb_fail(SPB_ERR_ARG, "unknown duplicate policy %d", policy);
    CK(cudaSetDevice(ctx->device));
    const u64 ncols = in->rank == 2 ? in->shape[1] : 1;
    const u64 cells = in->shape[0] * ncols;
    if (cells == 0) return SPB_OK;
    if (cells > (1ull << 33)) return spb_fail(SPB_ERR_TOO_LARGE, "spb_coo_to_dense: %llu cells", (ull)cells);
    Scratch ws(ctx);
    double *d;
    CKR(ws.get(&d, cells));
    CK(cudaMemsetAsync(d, 0, cells * sizeof(double), ctx->stream));  // ret = 0  (VectorCooArray.hpp:316)
    if (in->n) {
        // stable sort by cell, every entry kept (zeros too: REPLACE / LEAVE_ALONE see them), bounds checked
        const int so[2] = {0, 1};
        spb_coo *sorted = nullptr;
        CKR(consolidate_core(ctx, in, so, so, POLICY_KEEP_ALL, false, 0, &sorted, nullptr));
        ++ctx->launches, k_dense_fold<<<grid_for(sorted->n, 256, (u32)ctx->sm_count * 32), 256, 0, ctx->stream>>>(
            sorted->idx[0], in->rank == 2 ? sorted->idx[1] : nullptr, sorted->val, sorted->n, ncols, policy, d);
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        spb_coo_free(ctx, sorted);
        if (e != cudaSuccess) return spb_fail(SPB_ERR_CUDA, "spb_coo_to_dense: %s", cudaGetErrorString(e));
    }
    CK(cudaMemcpyAsync(dense, d, cells * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SPB_OK;
}

int spb_dense_to_coo(spb_ctx *ctx, int rank, const uint64_t *shape, const double *dense, spb_coo **out) {
    if (!ctx || !shape || !out || (rank != 1 && rank != 2)) return spb_fail(SPB_ERR_ARG, "spb_dense_to_coo: bad argument");
    CK(cudaSetDevice(ctx->device));
    const u64 ncols = rank == 2 ? shape[1] : 1;
    const u64 cells = shape[0] * ncols;
    if (cells && !dense) return spb_fail(SPB_ERR_ARG, "spb_dense_to_coo: null data pointer");
    if (cells > (1ull << 33)) return spb_fail(SPB_ERR_TOO_LARGE, "spb_dense_to_coo: %llu cells", (ull)cells);
    u64 n = 0;
    Scratch ws(ctx);
    double *d = nullptr;
    unsigned char *keep = nullptr;
    u64 *slot = nullptr;
    const u32 cap = (u32)ctx->sm_count * 32;
    if (cells) {
        CKR(ws.get(&d, cells));
        CKR(ws.get(&keep, cells));
        CKR(ws.get(&slot, cells + 1));
        CK(cudaMemcpyAsync(d, dense, cells * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        ++ctx->launches, k_dense_flags<<<grid_for(cells, 256, cap), 256, 0, ctx->stream>>>(d, cells, keep);
        CKR((exclusive_scan<unsigned char, u64>(ctx, ws, keep, slot, cells)));
        CK(cudaMemcpyAsync(&n, slot + cells, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    if (n >= (1ull << 31)) return spb_fail(SPB_ERR_TOO_LARGE, "spb_dense_to_coo: %llu entries; a VectorCooArray holds < 2^31", (ull)n);
    CKR(coo_new(ctx, rank, shape, n, true, out));
    spb_coo *r = *out;
    if (n) {
        ++ctx->launches, k_dense_compact<<<grid_for(cells, 256, cap), 256, 0, ctx->stream>>>(d, cells, ncols, keep, slot, r->idx[0],
                                                                                     rank == 2 ? r->idx[1] : nullptr, r->val);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return SPB_OK;  // edit mode, not flagged sorted (to_sparse only add()s)
}

int spb_dim_beginnings(spb_ctx *ctx, const spb_coo *a, uint64_t *out, uint64_t cap, uint64_t *count) {
    if (!ctx || !a || !count) return spb_fail(SPB_ERR_ARG, "spb_dim_beginnings: null argument");
    if (a->sort_order[0] < 0)
        return spb_fail(SPB_ERR_NOT_SORTED, "dim_beginnings() required the VectorCooArray is sorted first.");
    *count = 0;
    if (a->n == 0) return SPB_OK;  // algorithm.hpp:89: empty array, empty list
    CK(cudaSetDevice(ctx->device));
    RowIndex ri;
    CKR(build_row_index(ctx, a, &ri));
    *count = (u64)ri.nrows + 1;
    u64 take = *count < cap ? *count : cap;
    if (out && take) {
        std::vector<u32> h(take);
        CK(cudaMemcpyAsync(h.data(), ri.start, take * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        for (u64 i = 0; i < take; ++i) out[i] = h[i];
    }
    return SPB_OK;
}

static int scale_ok(const spb_coo *s, const char *name) {
    if (s && s->rank != 1) return spb_fail(SPB_ERR_ARG, "%s must be a rank-1 array", name);
    return 0;
}

int spb_multiply_mm_prepared(spb_ctx *ctx, double C, const spb_coo *si, const spb_coo *A, int a_row_dim,
                             const spb_coo *sj, const spb_coo *B, int b_inner_dim, const spb_coo *sk,
                             spb_coo **out, spb_mm_stats *stats) {
    if (!ctx || !A || !B || !out) return spb_fail(SPB_ERR_ARG, "spb_multiply_mm_prepared: null argument");
    if (A->rank != 2 || B->rank != 2) return spb_fail(SPB_ERR_ARG, "A and B must be rank-2 arrays");
    if ((a_row_dim | 1) != 1 || (b_inner_dim | 1) != 1) return spb_fail(SPB_ERR_ARG, "dimension must be 0 or 1");
    CKR(scale_ok(si, "scalei")); CKR(scale_ok(sj, "scalej")); CKR(scale_ok(sk, "scalek"));
    if (A->n && (!A->idx[0] || !A->idx[1])) return spb_fail(SPB_ERR_ARG, "A must be a full COO array");
    if (A->sort_order[0] != a_row_dim || B->sort_order[0] != b_inner_dim)
        return spb_fail(SPB_ERR_NOT_SORTED, "prepared operands must be consolidated by (row, inner) and (inner, col)");
    CK(cudaSetDevice(ctx->device));
    if (stats) memset(stats, 0, sizeof *stats);
    const u64 shape[2] = {A->shape[a_row_dim], B->shape[1 - b_inner_dim]};
    if (A->shape[1 - a_row_dim] != B->shape[b_inner_dim])
        return spb_fail(SPB_ERR_INNER_DIM, "Inner dimensions for A (%ld) and B (%ld) must match!",
                        (long)A->shape[1 - a_row_dim], (long)B->shape[b_inner_dim]);
    spb_coo *r = nullptr;
    CKR(coo_new(ctx, 2, shape, 0, false, &r));
    r->owned = true;
    *out = r;
    if (C == 0.0 || (si && si->n == 0) || A->n == 0 || (sj && sj->n == 0) || B->n == 0 || (sk && sk->n == 0))
        return SPB_OK;
    Timer tm(ctx->stream);
    const int t0 = tm.mark();
    int rc = multiply_core(ctx, C, si, A, a_row_dim, sj, B, b_inner_dim, sk, r, stats, tm, t0);
    if (rc) { spb_coo_free(ctx, r); *out = nullptr; }
    return rc;
}

int spb_multiply_mm(spb_ctx *ctx, double C, const spb_coo *si, const spb_coo *A, char tA, const spb_coo *sj,
                    const spb_coo *B, char tB, const spb_coo *sk, int policy, int zero_nan, spb_coo **out,
                    spb_mm_stats *stats) {
    if (!ctx || !A || !B || !out) return spb_fail(SPB_ERR_ARG, "spb_multiply_mm: null argument");
    if (A->rank != 2 || B->rank != 2) return spb_fail(SPB_ERR_ARG, "A and B must be rank-2 arrays");
    if (policy < 0 || policy > 2) return spb_fail(SPB_ERR_ARG, "unknown duplicate policy %d", policy);
    CKR(scale_ok(si, "scalei")); CKR(scale_ok(sj, "scalej")); CKR(scale_ok(sk, "scalek"));
    CK(cudaSetDevice(ctx->device));
    if (stats) memset(stats, 0, sizeof *stats);
    // multiply_sparse.hpp:167-169
    const int a_so[2] = {tA == 'T' ? 1 : 0, tA == 'T' ? 0 : 1};
    const int b_so[2] = {tB == 'T' ? 0 : 1, tB == 'T' ? 1 : 0};  // the reference's order: (col, inner)
    const int b_mine[2] = {b_so[1], b_so[0]};                      // ours: (inner, col)
    const u64 shape[2] = {A->shape[a_so[0]], B->shape[b_so[0]]};
    if (A->shape[a_so[1]] != B->shape[b_so[1]])  // :172-174
        return spb_fail(SPB_ERR_INNER_DIM, "Inner dimensions for A (%ld) and B (%ld) must match!",
                        (long)A->shape[a_so[1]], (long)B->shape[b_so[1]]);
    spb_coo *r = nullptr;
    CKR(coo_new(ctx, 2, shape, 0, false, &r));
    r->owned = true;
    *out = r;
    // :178-184
    if (C == 0.0 || (si && si->n == 0) || A->n == 0 || (sj && sj->n == 0) || B->n == 0 || (sk && sk->n == 0))
        return SPB_OK;
    Timer tm(ctx->stream);
    const int t0 = tm.mark();
    // Consolidate<> (algorithm.hpp:354-369): reuse an operand already flagged sorted in the needed order
    spb_coo *Ac = nullptr, *Bc = nullptr;
    int rc = 0;
    const spb_coo *Ause = A, *Buse = B;
    if (!(A->sort_order[0] == a_so[0] && A->sort_order[1] == a_so[1])) {
        rc = consolidate_core(ctx, A, a_so, a_so, policy, true, zero_nan, &Ac, nullptr);
        Ause = Ac;
    }
    if (!rc) {
        if (B->sort_order[0] == b_so[0] && B->sort_order[1] == b_so[1]) {
            // the reference would use B as stored: re-bucket by inner index, keep every entry
            rc = consolidate_core(ctx, B, b_mine, b_so, POLICY_KEEP_ALL, false, 0, &Bc, nullptr);
        } else {
            rc = consolidate_core(ctx, B, b_mine, b_so, policy, true, zero_nan, &Bc, nullptr);
        }
        Buse = Bc;
    }
    if (!rc && Ause->n && Buse->n)
        rc = multiply_core(ctx, C, si, Ause, a_so[0], sj, Buse, b_mine[0], sk, r, stats, tm, t0);
    spb_coo_free(ctx, Ac);
    spb_coo_free(ctx, Bc);
    if (rc) { spb_coo_free(ctx, r); *out = nullptr; }
    return rc;
}

int spb_multiply_mv(spb_ctx *ctx, double C, const spb_coo *si, const spb_coo *A, char tA, const spb_coo *sj,
                    const spb_coo *V, int policy, int zero_nan, spb_coo **out) {
    if (!ctx || !A || !V || !out) return spb_fail(SPB_ERR_ARG, "spb_multiply_mv: null argument");
    if (A->rank != 2 || V->rank != 1) return spb_fail(SPB_ERR_ARG, "A must be rank 2 and V rank 1");
    if (policy < 0 || policy > 2) return spb_fail(SPB_ERR_ARG, "unknown duplicate policy %d", policy);
    CKR(scale_ok(si, "scalei")); CKR(scale_ok(sj, "scalej"));
    CK(cudaSetDevice(ctx->device));
    const int a_so[2] = {tA == 'T' ? 1 : 0, tA == 'T' ? 0 : 1};  // multiply_sparse.hpp:294
    const u64 shape[1] = {A->shape[a_so[0]]};
    if (A->shape[a_so[1]] != V->shape[0])  // :298-300
        return spb_fail(SPB_ERR_INNER_DIM, "Inner dimensions for A (%ld) and V (%ld) must match!",
                        (long)A->shape[a_so[1]], (long)V->shape[0]);
    spb_coo *r = nullptr;
    CKR(coo_new(ctx, 1, shape, 0, false, &r));
    r->owned = true;
    *out = r;
    if (C == 0.0 || (si && si->n == 0) || A->n == 0 || (sj && sj->n == 0) || V->n == 0) return SPB_OK;  // :304-309
    spb_coo *Ac = nullptr, *Vc = nullptr;
    const spb_coo *Ause = A, *Vuse = V;
    const int v_so[2] = {0, 0};
    int rc = 0;
    if (!(A->sort_order[0] == a_so[0] && A->sort_order[1] == a_so[1])) {
        rc = consolidate_core(ctx, A, a_so, a_so, policy, true, zero_nan, &Ac, nullptr);  // :312
        Ause = Ac;
    }
    if (!rc && V->sort_order[0] != 0) {
        rc = consolidate_core(ctx, V, v_so, v_so, policy, true, zero_nan, &Vc, nullptr);  // :313
        Vuse = Vc;
    }
    if (!rc && Ause->n) {
        Scratch ws(ctx);
        const u64 m_rows = A->shape[a_so[0]], n_inner = A->shape[a_so[1]];
        MMOperands m;
        memset(&m, 0, sizeof m);
        m.C = C;
        m.a_j = Ause->idx[a_so[1]]; m.a_val = Ause->val; m.nnz_a = (u32)Ause->n;
        RowIndex ri;
        rc = build_row_index(ctx, Ause, &ri);
        double *d, *vd, *row_val;
        unsigned char *mask, *vmask, *row_keep;
        u32 *slot, *bad_vec = nullptr;
        if (!rc) {
            m.arow_id = ri.id; m.arow_start = ri.start; m.nrows = ri.nrows;
            rc = ws.zeroed(&bad_vec, 1);
            if (!rc && si) { rc = densify(ctx, ws, si, m_rows, &d, nullptr, bad_vec); m.si = d; }
        }
        if (!rc && sj) { rc = densify(ctx, ws, sj, n_inner, &d, &mask, bad_vec); m.sj = d; m.sj_mask = mask; }
        if (!rc) rc = densify(ctx, ws, Vuse, n_inner, &vd, &vmask, bad_vec);
        if (!rc) rc = ws.get(&row_val, ri.nrows);
        if (!rc) rc = ws.get(&row_keep, ri.nrows);
        if (!rc) rc = ws.get(&slot, (u64)ri.nrows + 1);
        if (!rc) {
            const u32 cap = (u32)ctx->sm_count * 32;
            ++ctx->launches, k_mv_rows<<<grid_for(ri.nrows, 256, cap), 256, 0, ctx->stream>>>(m, vd, vmask, row_val, row_keep);
            rc = exclusive_scan<unsigned char, u32>(ctx, ws, row_keep, slot, ri.nrows);
            u32 nout = 0, h_bad = 0;
            if (!rc) {
                cudaMemcpyAsync(&nout, slot + ri.nrows, sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream);
                cudaMemcpyAsync(&h_bad, bad_vec, sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream);
                if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = spb_fail(SPB_ERR_CUDA, "multiply_mv: %s", cudaGetErrorString(cudaGetLastError()));
                else if (h_bad) rc = bad_scale_vector();
            }
            if (!rc) {
                size_t cnt = nout ? nout : 1;
                if (ctx->pool.alloc((void **)&r->idx[0], cnt * sizeof(i32)) != cudaSuccess ||
                    ctx->pool.alloc((void **)&r->val, cnt * sizeof(double)) != cudaSuccess)
                    rc = spb_fail(SPB_ERR_CUDA, "multiply_mv: out of device memory");
            }
            if (!rc) {
                r->n = nout;
                if (nout) ++ctx->launches, k_mv_emit<<<grid_for(ri.nrows, 256, cap), 256, 0, ctx->stream>>>(ri.nrows, ri.id, row_val, row_keep, slot, r->idx[0], r->val);
                if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = spb_fail(SPB_ERR_CUDA, "multiply_mv: %s", cudaGetErrorString(cudaGetLastError()));
            }
        }
    }
    spb_coo_free(ctx, Ac);
    spb_coo_free(ctx, Vc);
    if (rc) { spb_coo_free(ctx, r); *out = nullptr; }
    return rc;
}

}  // extern "C"

// ---- consolidate with a fixed index pattern ----------------------------------------------------------------------------
// The pattern is sorted once (cons_plan.cuh); a run gathers the new values into that order, dropping what consolidate()
// drops, and hands the kept pairs to the duplicate-reduce that sort_reduce runs after its passes.  12 bytes of device memory
// per entry, from the context's pool.
struct spb_cons_plan {
    spb_ctx *ctx;
    int rank;
    u64 shape[2];
    int so[2];
    u64 n;
    int bits_lo, key_bits;
    u64 *keys;   // [n] packed keys (idx[so[0]] << bits_lo) | idx[so[1]], in stable sorted order
    u32 *perm;   // [n] sorted position -> entry number
};

// n values given to a plan run: device memory is read in place; host memory is staged as spb_coo_upload stages it
static int device_values(spb_ctx *ctx, Scratch &ws, const double *val, u64 n, const char *what, const double **dval) {
    *dval = val;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, val) != cudaSuccess) { cudaGetLastError(); at.type = cudaMemoryTypeUnregistered; }
    if (at.type == cudaMemoryTypeDevice && at.device != ctx->device)
        return spb_fail(SPB_ERR_ARG, "%s: values on device %d, the plan's context is on device %d", what, at.device, ctx->device);
    if (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) {
        double *staged;
        CKR(ws.get(&staged, n));
        const XferJob job = {staged, const_cast<double *>(val), (size_t)n * sizeof(double)};
        CKR(staged_copy(ctx, &job, 1, true));
        *dval = staged;
    }
    return 0;
}

// the reduce of the kept pairs into r (allocated for plan->n entries); statistics as spb_consolidate_stats describes
static int cons_plan_run(spb_cons_plan *plan, const double *dval, int policy, int zero_nan, spb_coo *r,
                         spb_consolidate_stats *st) {
    spb_ctx *ctx = plan->ctx;
    const u32 n = (u32)plan->n;
    Scratch ws(ctx);
    Timer tm(ctx->stream);
    const int t0 = tm.mark();
    u32 *counters, *tickets, *bound = nullptr;   // counters: [0] kept, [2] out count, [3] long runs, [4] rows
    u64 *gstate, *kA;
    double *vA;
    const u32 tiles = (u32)div_up(n, CP_TILE);
    CKR(ws.zeroed(&counters, 8));
    CKR(ws.zeroed(&tickets, 2));
    CKR(ws.zeroed(&gstate, tiles));
    CKR(ws.get(&kA, n));
    CKR(ws.get(&vA, n));
    if (zero_nan) {
        CKR(ws.get(&bound, 1));
        CK(cudaMemsetAsync(bound, 0xFF, sizeof(u32), ctx->stream));
        const u32 grid = tiles < (u32)ctx->sm_count * 2 ? tiles : (u32)ctx->sm_count * 2;
        ++ctx->launches, k_plan_first_kept<<<grid, CP_THREADS, 0, ctx->stream>>>(plan->perm, dval, n, tickets + 1, bound);
    }
    PlanGatherArgs ga;
    ga.keys = plan->keys; ga.perm = plan->perm; ga.val = dval; ga.n = n; ga.bound = bound;
    ga.keys_out = kA; ga.vals_out = vA; ga.n_kept = counters; ga.state = gstate; ga.ticket = tickets;
    ++ctx->launches, k_plan_gather<<<tiles, CP_THREADS, 0, ctx->stream>>>(ga);
    CK(cudaGetLastError());
    const int t1 = tm.mark();

    // the reduce pass sort_reduce runs where no in-row sort counted the heads: a block per tile, placed by a look-back (the
    // warp-per-tile look-back variant measured slower, DESIGN.md section 3)
    const u32 rtiles = (u32)div_up(n, RK_TILE);
    ReduceArgs ra;
    memset(&ra, 0, sizeof ra);
    ra.keys = kA; ra.vals = vA; ra.n_ptr = counters; ra.bits_lo = plan->bits_lo; ra.policy = policy;
    ra.out_hi = r->idx[plan->so[0]]; ra.out_lo = plan->rank > 1 ? r->idx[plan->so[1]] : nullptr; ra.out_val = r->val;
    ra.out_count = counters + 2;
    CKR(ws.zeroed(&ra.state, rtiles));
    CKR(ws.zeroed(&ra.ticket, 1));
    ra.long_cap = n / RK_LONG_RUN + 1;
    CKR(ws.get(&ra.long_list, 2ull * ra.long_cap));
    ra.long_count = counters + 3;
    ra.row_start = r->row_start; ra.row_id = r->row_id; ra.row_count = counters + 4;
    ++ctx->launches, k_reduce_by_key<MODE_CONSOLIDATE><<<rtiles, RK_THREADS, 0, ctx->stream>>>(ra);
    if (policy == POLICY_ADD || policy == POLICY_REPLACE)
        ++ctx->launches, k_long_runs<<<(u32)ctx->sm_count * 4, 256, 0, ctx->stream>>>(ra);
    CK(cudaGetLastError());
    const int t2 = tm.mark();

    u32 h[8];
    CK(cudaMemcpyAsync(h, counters, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    r->n = h[2];
    if (plan->rank == 2) {
        r->nrows = h[4];
        r->rows_valid = true;
        if (h[2] == 0) { const u32 z = 0; CK(cudaMemcpyAsync(r->row_start, &z, sizeof z, cudaMemcpyHostToDevice, ctx->stream)); CK(cudaStreamSynchronize(ctx->stream)); }
    }
    if (st) {
        st->n_in = n; st->n_kept = h[0]; st->n_out = h[2];
        st->key_bits = plan->key_bits; st->passes = 0; st->digit_bits = 0;
        st->ms_sort = tm.ms(t0, t1); st->ms_reduce = tm.ms(t1, t2); st->ms_total = tm.ms(t0, t2);
        st->ms_pass = 0.f;
    }
    return 0;
}

extern "C" {

int spb_consolidate_plan_create(spb_ctx *ctx, const spb_coo *in, const int *sort_order, spb_cons_plan **out,
                                uint64_t *n_runs) {
    if (!ctx || !in || !out) return spb_fail(SPB_ERR_ARG, "spb_consolidate_plan_create: null argument");
    CKR(check_order(in, sort_order, "spb_consolidate_plan_create"));
    if (in->n >= (1ull << 31)) return spb_fail(SPB_ERR_TOO_LARGE, "%llu entries: one array holds fewer than 2^31 (the reference's own cap, algorithm.hpp:419)", (ull)in->n);
    CK(cudaSetDevice(ctx->device));
    spb_cons_plan *p = new spb_cons_plan();
    p->ctx = ctx;
    p->rank = in->rank;
    p->shape[0] = in->shape[0]; p->shape[1] = in->shape[1];
    p->so[0] = sort_order[0]; p->so[1] = in->rank > 1 ? sort_order[1] : 0;
    p->n = in->n;
    p->bits_lo = in->rank > 1 ? bits_for(in->shape[p->so[1]]) : 0;
    p->key_bits = bits_for(in->shape[p->so[0]]) + p->bits_lo;
    p->keys = nullptr; p->perm = nullptr;
    u32 runs = 0;
    if (in->n) {
        // what spb_sorted_permutation does: a stable sort with the entry numbers as payload, nothing dropped or merged
        Scratch ws(ctx);
        double *iota;
        u32 *cnt;
        int rc = ws.get(&iota, in->n);
        if (!rc) rc = ws.zeroed(&cnt, 1);
        spb_coo *sorted = nullptr;
        if (!rc) {
            ++ctx->launches, k_iota_bits<<<grid_for(in->n, 256, 1u << 16), 256, 0, ctx->stream>>>(in->n, iota);
            spb_coo tmp = *in;
            tmp.val = iota;
            tmp.owned = false;
            rc = consolidate_core(ctx, &tmp, p->so, p->so, POLICY_KEEP_ALL, false, 0, &sorted, nullptr);
        }
        if (!rc && sorted->n != in->n)
            rc = spb_fail(SPB_ERR_CUDA, "spb_consolidate_plan_create: lost entries (%llu of %llu)", (ull)sorted->n, (ull)in->n);
        if (!rc && (ctx->pool.alloc((void **)&p->keys, in->n * sizeof(u64)) != cudaSuccess ||
                    ctx->pool.alloc((void **)&p->perm, in->n * sizeof(u32)) != cudaSuccess))
            rc = spb_fail(SPB_ERR_CUDA, "spb_consolidate_plan_create: out of device memory (%llu entries)", (ull)in->n);
        if (!rc) {
            ++ctx->launches, k_plan_pack<<<grid_for(in->n, 256, (u32)ctx->sm_count * 16), 256, 0, ctx->stream>>>(
                sorted->idx[p->so[0]], in->rank > 1 ? sorted->idx[p->so[1]] : nullptr, sorted->val, (u32)in->n, p->bits_lo,
                p->keys, p->perm, cnt);
            cudaError_t e = cudaGetLastError();
            if (e == cudaSuccess) e = cudaMemcpyAsync(&runs, cnt, sizeof runs, cudaMemcpyDeviceToHost, ctx->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
            if (e != cudaSuccess) rc = spb_fail(SPB_ERR_CUDA, "spb_consolidate_plan_create: %s", cudaGetErrorString(e));
        }
        spb_coo_free(ctx, sorted);
        if (rc) {
            spb_consolidate_plan_destroy(p);
            return rc;
        }
    }
    *out = p;
    if (n_runs) *n_runs = runs;
    return SPB_OK;
}

int spb_consolidate_plan_run(spb_cons_plan *plan, const double *val, int policy, int zero_nan, spb_coo **out,
                             spb_consolidate_stats *stats) {
    if (!plan || !out) return spb_fail(SPB_ERR_ARG, "spb_consolidate_plan_run: null argument");
    if (plan->n && !val) return spb_fail(SPB_ERR_ARG, "spb_consolidate_plan_run: null value pointer");
    if (policy < 0 || policy > 2) return spb_fail(SPB_ERR_ARG, "unknown duplicate policy %d", policy);
    if ((uintptr_t)val & 7u) return spb_fail(SPB_ERR_ARG, "spb_consolidate_plan_run: value pointer is not 8-byte aligned");
    spb_ctx *ctx = plan->ctx;
    CK(cudaSetDevice(ctx->device));
    if (stats) memset(stats, 0, sizeof *stats);
    Scratch ws(ctx);
    const double *dval = val;
    if (plan->n) CKR(device_values(ctx, ws, val, plan->n, "spb_consolidate_plan_run", &dval));
    spb_coo *r = nullptr;
    CKR(coo_new(ctx, plan->rank, plan->shape, plan->n, true, &r));
    set_order(r, plan->so);
    if (plan->n == 0) { *out = r; return SPB_OK; }  // algorithm.hpp:263,318
    int rc = 0;
    if (plan->rank == 2) {  // the reduce pass also emits the compressed row starts of its output
        const u64 ext = plan->shape[plan->so[0]];
        const u64 cap = (plan->n < ext ? plan->n : ext) + 1;
        if (ctx->pool.alloc((void **)&r->row_start, cap * sizeof(u32)) != cudaSuccess ||
            ctx->pool.alloc((void **)&r->row_id, cap * sizeof(i32)) != cudaSuccess)
            rc = spb_fail(SPB_ERR_CUDA, "out of device memory");
    }
    if (!rc) rc = cons_plan_run(plan, dval, policy, zero_nan, r, stats);
    if (rc) { spb_coo_free(ctx, r); return rc; }
    *out = r;
    return SPB_OK;
}

int spb_consolidate_plan_destroy(spb_cons_plan *plan) {
    if (!plan) return SPB_OK;
    plan->ctx->pool.release(plan->keys);
    plan->ctx->pool.release(plan->perm);
    delete plan;
    return SPB_OK;
}

}  // extern "C"

// ---- multiply with a fixed operand pattern -----------------------------------------------------------------------------
// Everything spb_multiply_mm does that depends only on the operands' indices and the scale vectors -- the consolidations'
// sorts, the row index of A, B's dense pointer, the densified scale vectors, the whole symbolic phase -- is done once at
// creation.  A run folds the new values into one slot per run of equal indices (mm_pattern.cuh) and, when no run came out
// empty, runs only the numeric kernels on the placement the creation made.  When a run is empty the operands' patterns are
// smaller than the plan's: the non-empty runs are compacted -- exactly what spb_multiply_mm's consolidations return -- and the
// whole multiply runs on them.
enum { PO_FOLD = 0, PO_GATHER = 1, PO_AS_GIVEN = 2 };
struct PatternOperand {
    int mode;                       // PO_FOLD: consolidated by spb_multiply_mm; PO_GATHER: B flagged in the reference's order
                                    // (re-bucketed, every entry kept); PO_AS_GIVEN: A flagged (row, inner), used as it is
    u32 n = 0, runs = 0;            // entries of the value array; entries of `full`
    u32 *perm = nullptr;            // [n] sorted position -> entry number (PO_FOLD, PO_GATHER)
    u32 *off = nullptr;             // [runs + 1] first sorted position of every run (PO_FOLD)
    u32 *ref_pos = nullptr;         // [n] B with zero_nan: sorted entry -> position in the reference's order (PO_FOLD)
    unsigned char *live = nullptr;  // [runs] set by a fold (PO_FOLD)
    spb_coo *full = nullptr;        // the operand with every run present, one entry per run; full->val holds the folded values
};

struct spb_mm_pattern {
    spb_ctx *ctx;
    double C;
    int policy, zero_nan;
    u64 shape[2];
    bool empty;                     // the product is empty whatever the values (C = 0, an empty scale vector or operand)
    int a_row_dim, b_inner_dim;
    spb_coo *si = nullptr, *sj = nullptr, *sk = nullptr;   // copies of the scale vectors
    PatternOperand A, B;
    Scratch *sym = nullptr;         // device memory of the symbolic phase
    MmState s;
};

// Sorts `in` by `so` once (stable, every entry kept, the entry numbers as payload).  PO_FOLD: the run offsets and the
// consolidated index vectors of the full pattern, and with ref_so the reference positions; PO_GATHER: the sorted array itself.
static int pattern_operand(spb_ctx *ctx, const spb_coo *in, const int *so, const int *ref_so, PatternOperand &op) {
    const u32 n = (u32)in->n;
    const u32 grid = (u32)ctx->sm_count * 16;
    op.n = n;
    Scratch ws(ctx);
    double *iota;
    CKR(ws.get(&iota, n));
    ++ctx->launches, k_iota_bits<<<grid_for(n, 256, 1u << 16), 256, 0, ctx->stream>>>(n, iota);
    spb_coo tmp = *in;
    tmp.val = iota;
    tmp.owned = false;
    spb_coo *sorted = nullptr;
    CKR(consolidate_core(ctx, &tmp, so, so, POLICY_KEEP_ALL, false, 0, &sorted, nullptr));
    if (sorted->n != n) {
        spb_coo_free(ctx, sorted);
        return spb_fail(SPB_ERR_CUDA, "spb_mm_pattern_create: lost entries (%llu of %u)", (ull)sorted->n, n);
    }
    const i32 *hi = sorted->idx[so[0]], *lo = sorted->idx[so[1]];
    unsigned char *head;
    CKR(ws.get(&head, n));
    CK(ctx->pool.alloc((void **)&op.perm, (u64)n * sizeof(u32)));
    ++ctx->launches, k_pattern_heads<<<grid_for(n, 256, grid), 256, 0, ctx->stream>>>(hi, lo, sorted->val, n, op.perm, head);
    if (op.mode == PO_GATHER) {
        op.runs = n;
        op.full = sorted;   // its values (the entry numbers) are overwritten by every run
        return 0;
    }
    u64 *slot;
    CKR(ws.get(&slot, (u64)n + 1));
    CKR((exclusive_scan<unsigned char, u64>(ctx, ws, head, slot, n)));
    u64 runs = 0;
    CK(cudaMemcpyAsync(&runs, slot + n, sizeof runs, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    op.runs = (u32)runs;
    int rc = coo_new(ctx, 2, in->shape, runs, true, &op.full);
    if (!rc) {
        set_order(op.full, so);
        if (ctx->pool.alloc((void **)&op.off, (runs + 1) * sizeof(u32)) != cudaSuccess ||
            ctx->pool.alloc((void **)&op.live, runs) != cudaSuccess)
            rc = spb_fail(SPB_ERR_CUDA, "spb_mm_pattern_create: out of device memory (%llu runs)", (ull)runs);
    }
    if (!rc) {
        ++ctx->launches, k_pattern_runs<<<grid_for(n, 256, grid), 256, 0, ctx->stream>>>(hi, lo, head, slot, n, op.off,
                                                                                         op.full->idx[so[0]], op.full->idx[so[1]]);
        if (cudaGetLastError() != cudaSuccess) rc = spb_fail(SPB_ERR_CUDA, "spb_mm_pattern_create: launch failed");
    }
    spb_coo_free(ctx, sorted);
    if (rc || !ref_so) return rc;
    // the reference's order: sorted the same way; inv[entry] = its position there
    spb_coo *ref = nullptr;
    CKR(consolidate_core(ctx, &tmp, ref_so, ref_so, POLICY_KEEP_ALL, false, 0, &ref, nullptr));
    u32 *inv;
    rc = ws.get(&inv, n);
    if (!rc && ctx->pool.alloc((void **)&op.ref_pos, (u64)n * sizeof(u32)) != cudaSuccess)
        rc = spb_fail(SPB_ERR_CUDA, "spb_mm_pattern_create: out of device memory (%u entries)", n);
    if (!rc) {
        ++ctx->launches, k_pattern_invert<<<grid_for(n, 256, grid), 256, 0, ctx->stream>>>(ref->val, n, inv);
        ++ctx->launches, k_pattern_ref_pos<<<grid_for(n, 256, grid), 256, 0, ctx->stream>>>(op.perm, inv, n, op.ref_pos);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(ctx->stream));   // inv dies with ws
    }
    spb_coo_free(ctx, ref);
    return rc;
}

static void pattern_operand_free(spb_ctx *ctx, PatternOperand &op) {
    ctx->pool.release(op.perm); ctx->pool.release(op.off); ctx->pool.release(op.ref_pos); ctx->pool.release(op.live);
    spb_coo_free(ctx, op.full);
    op.perm = op.off = op.ref_pos = nullptr; op.live = nullptr; op.full = nullptr;
}

// A run's values for one operand: folded into op.full->val (PO_FOLD; counters[0] += runs left empty, counters[1]: long runs),
// gathered into it (PO_GATHER), or nothing to do (PO_AS_GIVEN).
static int pattern_fold(spb_ctx *ctx, Scratch &ws, PatternOperand &op, const double *val, int policy, int zero_nan, u32 *counters) {
    if (op.mode == PO_AS_GIVEN) return 0;
    if (op.mode == PO_GATHER) {
        ++ctx->launches, k_pattern_gather<<<grid_for(op.n, 256, (u32)ctx->sm_count * 16), 256, 0, ctx->stream>>>(op.perm, val, op.n, op.full->val);
        CK(cudaGetLastError());
        return 0;
    }
    PatternFold f;
    f.perm = op.perm; f.off = op.off; f.ref_pos = op.ref_pos; f.val = val; f.bound = nullptr;
    f.runs = op.runs; f.policy = policy; f.out = op.full->val; f.live = op.live;
    f.empty = counters; f.long_count = counters + 1;
    f.long_cap = op.n / PF_LONG_RUN + 1;
    CKR(ws.get(&f.long_list, f.long_cap));
    if (zero_nan) {
        u32 *bound;
        CKR(ws.get(&bound, 1));
        CK(cudaMemsetAsync(bound, 0xFF, sizeof(u32), ctx->stream));
        if (op.ref_pos) {
            ++ctx->launches, k_pattern_ref_bound<<<grid_for(op.n, 256, (u32)ctx->sm_count * 8), 256, 0, ctx->stream>>>(op.perm, op.ref_pos, val, op.n, bound);
        } else {   // the reference sorts as the plan does: the first kept sorted position, found from the front
            u32 *ticket;
            CKR(ws.zeroed(&ticket, 1));
            const u32 tiles = (u32)div_up(op.n, CP_TILE);
            const u32 grid = tiles < (u32)ctx->sm_count * 2 ? tiles : (u32)ctx->sm_count * 2;
            ++ctx->launches, k_plan_first_kept<<<grid, CP_THREADS, 0, ctx->stream>>>(op.perm, val, op.n, ticket, bound);
        }
        f.bound = bound;
    }
    ++ctx->launches, k_pattern_fold<<<grid_for(op.runs, 256, (u32)ctx->sm_count * 16), 256, 0, ctx->stream>>>(f);
    ++ctx->launches, k_pattern_fold_long<<<(u32)ctx->sm_count * 4, 256, 0, ctx->stream>>>(f);
    CK(cudaGetLastError());
    return 0;
}

// The non-empty runs of a folded operand, compacted: what spb_multiply_mm's consolidation returns for these values.
static int pattern_compact(spb_ctx *ctx, Scratch &ws, const PatternOperand &op, u64 kept, spb_coo **out) {
    spb_coo *r = nullptr;
    CKR(coo_new(ctx, 2, op.full->shape, kept, true, &r));
    set_order(r, op.full->sort_order);
    u64 *slot;
    int rc = ws.get(&slot, (u64)op.runs + 1);
    if (!rc) rc = exclusive_scan<unsigned char, u64>(ctx, ws, op.live, slot, op.runs);
    if (!rc) {
        ++ctx->launches, k_compact_entries<<<grid_for(op.runs, 256, (u32)ctx->sm_count * 32), 256, 0, ctx->stream>>>(
            op.runs, op.live, slot, op.full->idx[0], op.full->idx[1], op.full->val, r->idx[0], r->idx[1], r->val);
        if (cudaGetLastError() != cudaSuccess) rc = spb_fail(SPB_ERR_CUDA, "pattern compaction: launch failed");
    }
    if (rc) { spb_coo_free(ctx, r); return rc; }
    *out = r;
    return 0;
}

extern "C" {

int spb_mm_pattern_destroy(spb_mm_pattern *plan) {
    if (!plan) return SPB_OK;
    spb_ctx *ctx = plan->ctx;
    delete plan->sym;
    pattern_operand_free(ctx, plan->A);
    pattern_operand_free(ctx, plan->B);
    spb_coo_free(ctx, plan->si); spb_coo_free(ctx, plan->sj); spb_coo_free(ctx, plan->sk);
    delete plan;
    return SPB_OK;
}

int spb_mm_pattern_create(spb_ctx *ctx, double C, const spb_coo *si, const spb_coo *A, char tA, const spb_coo *sj,
                          const spb_coo *B, char tB, const spb_coo *sk, int policy, int zero_nan, spb_mm_pattern **out,
                          uint64_t *nnz_bound) {
    if (!ctx || !A || !B || !out) return spb_fail(SPB_ERR_ARG, "spb_mm_pattern_create: null argument");
    if (A->rank != 2 || B->rank != 2) return spb_fail(SPB_ERR_ARG, "A and B must be rank-2 arrays");
    if (policy < 0 || policy > 2) return spb_fail(SPB_ERR_ARG, "unknown duplicate policy %d", policy);
    CKR(scale_ok(si, "scalei")); CKR(scale_ok(sj, "scalej")); CKR(scale_ok(sk, "scalek"));
    if ((A->n && (!A->idx[0] || !A->idx[1])) || (B->n && (!B->idx[0] || !B->idx[1])))
        return spb_fail(SPB_ERR_ARG, "spb_mm_pattern_create: A and B must be full COO arrays");
    if (A->n >= (1ull << 31) || B->n >= (1ull << 31))
        return spb_fail(SPB_ERR_TOO_LARGE, "one array holds fewer than 2^31 entries (the reference's own cap, algorithm.hpp:419)");
    CK(cudaSetDevice(ctx->device));
    const int a_so[2] = {tA == 'T' ? 1 : 0, tA == 'T' ? 0 : 1};
    const int b_so[2] = {tB == 'T' ? 0 : 1, tB == 'T' ? 1 : 0};   // the reference's order: (col, inner)
    const int b_mine[2] = {b_so[1], b_so[0]};                       // ours: (inner, col)
    if (A->shape[a_so[1]] != B->shape[b_so[1]])
        return spb_fail(SPB_ERR_INNER_DIM, "Inner dimensions for A (%ld) and B (%ld) must match!",
                        (long)A->shape[a_so[1]], (long)B->shape[b_so[1]]);
    spb_mm_pattern *p = new spb_mm_pattern();
    p->ctx = ctx; p->C = C; p->policy = policy; p->zero_nan = zero_nan ? 1 : 0;
    p->shape[0] = A->shape[a_so[0]]; p->shape[1] = B->shape[b_so[0]];
    p->a_row_dim = a_so[0]; p->b_inner_dim = b_mine[0];
    p->A.mode = (A->sort_order[0] == a_so[0] && A->sort_order[1] == a_so[1]) ? PO_AS_GIVEN : PO_FOLD;
    p->B.mode = (B->sort_order[0] == b_so[0] && B->sort_order[1] == b_so[1]) ? PO_GATHER : PO_FOLD;
    p->A.n = (u32)A->n; p->B.n = (u32)B->n;
    p->empty = C == 0.0 || (si && si->n == 0) || A->n == 0 || (sj && sj->n == 0) || B->n == 0 || (sk && sk->n == 0);
    int rc = 0;
    if (!p->empty) {
        if (si) rc = spb_coo_copy(ctx, si, &p->si);
        if (!rc && sj) rc = spb_coo_copy(ctx, sj, &p->sj);
        if (!rc && sk) rc = spb_coo_copy(ctx, sk, &p->sk);
        if (!rc && p->A.mode == PO_AS_GIVEN) {
            rc = coo_new(ctx, 2, A->shape, A->n, true, &p->A.full);
            if (!rc) {
                set_order(p->A.full, a_so);
                p->A.runs = (u32)A->n;
                for (int k = 0; k < 2 && !rc; ++k)
                    if (cudaMemcpyAsync(p->A.full->idx[k], A->idx[k], A->n * sizeof(i32), cudaMemcpyDeviceToDevice, ctx->stream) != cudaSuccess)
                        rc = spb_fail(SPB_ERR_CUDA, "spb_mm_pattern_create: copy of A's indices failed");
            }
        } else if (!rc) {
            rc = pattern_operand(ctx, A, a_so, nullptr, p->A);
        }
        if (!rc) rc = pattern_operand(ctx, B, b_mine, (p->B.mode == PO_FOLD && zero_nan) ? b_so : nullptr, p->B);
        if (!rc) {
            p->sym = new Scratch(ctx);
            Timer tm(ctx->stream);
            const int t0 = tm.mark();
            bool done = false;
            rc = mm_symbolic(ctx, *p->sym, C, p->si, p->A.full, p->a_row_dim, p->sj, p->B.full, p->b_inner_dim, p->sk, nullptr,
                             nullptr, tm, t0, false, nullptr, true, p->s, &done);
            if (!rc && p->s.nnz_c >= (1ull << 31))
                rc = spb_fail(SPB_ERR_TOO_LARGE, "the pattern's product has %llu entries; a VectorCooArray holds < 2^31 (algorithm.hpp:419) -- "
                              "form it in row panels (spb_mm_plan_create)", (ull)p->s.nnz_c);
            int te, tsp;
            if (!rc && p->s.h_stats[5] && p->s.nnz_c) rc = mm_hash_items(ctx, *p->sym, p->s, tm, &te, &tsp);
            if (!rc && cudaStreamSynchronize(ctx->stream) != cudaSuccess)
                rc = spb_fail(SPB_ERR_CUDA, "spb_mm_pattern_create: %s", cudaGetErrorString(cudaGetLastError()));
            p->s.t_prep = -1;
        }
    }
    if (rc) { spb_mm_pattern_destroy(p); return rc; }
    *out = p;
    if (nnz_bound) *nnz_bound = p->empty ? 0 : p->s.nnz_c;
    return SPB_OK;
}

int spb_mm_pattern_run(spb_mm_pattern *plan, const double *a_val, const double *b_val, spb_coo **out,
                       spb_mm_pattern_stats *stats) {
    if (!plan || !out) return spb_fail(SPB_ERR_ARG, "spb_mm_pattern_run: null argument");
    if ((plan->A.n && !a_val) || (plan->B.n && !b_val)) return spb_fail(SPB_ERR_ARG, "spb_mm_pattern_run: null value pointer");
    if (((uintptr_t)a_val | (uintptr_t)b_val) & 7u) return spb_fail(SPB_ERR_ARG, "spb_mm_pattern_run: value pointer is not 8-byte aligned");
    spb_ctx *ctx = plan->ctx;
    CK(cudaSetDevice(ctx->device));
    if (stats) memset(stats, 0, sizeof *stats);
    spb_coo *r = nullptr;
    CKR(coo_new(ctx, 2, plan->shape, 0, false, &r));
    r->owned = true;
    if (plan->empty) { *out = r; return SPB_OK; }
    Scratch ws(ctx);
    const double *da = a_val, *db = b_val;
    int rc = device_values(ctx, ws, a_val, plan->A.n, "spb_mm_pattern_run", &da);
    if (!rc) {
        if (b_val == a_val) db = da;   // one array for both operands (A * diag(s) * A^T)
        else rc = device_values(ctx, ws, b_val, plan->B.n, "spb_mm_pattern_run", &db);
    }
    Timer tm(ctx->stream);
    const int t0 = tm.mark();
    u32 *counters = nullptr;   // [0] A: runs left empty, [1] A: long runs, [2..3] the same for B
    if (!rc) rc = ws.zeroed(&counters, 4);
    if (!rc) rc = pattern_fold(ctx, ws, plan->A, da, plan->policy, plan->zero_nan, counters);
    const int t1 = tm.mark();
    if (!rc) rc = pattern_fold(ctx, ws, plan->B, db, plan->policy, plan->zero_nan, counters + 2);
    const int t2 = tm.mark();
    u32 h[4] = {0, 0, 0, 0};
    if (!rc && cudaMemcpyAsync(h, counters, sizeof h, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) rc = spb_fail(SPB_ERR_CUDA, "counter read-back failed");
    if (!rc && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = spb_fail(SPB_ERR_CUDA, "%s", cudaGetErrorString(cudaGetLastError()));
    if (!rc && stats) {
        stats->fallback = (h[0] || h[2]) ? 1 : 0;
        stats->empty_runs_a = h[0]; stats->empty_runs_b = h[2];
        stats->ms_fold_a = tm.ms(t0, t1); stats->ms_fold_b = tm.ms(t1, t2);
    }
    spb_mm_stats *mst = stats ? &stats->mm : nullptr;
    if (!rc && !h[0] && !h[2]) {
        // fast path: every run present, the operands have the plan's pattern -- only the numeric kernels run
        MmState s = plan->s;
        s.m.a_val = plan->A.mode == PO_AS_GIVEN ? da : plan->A.full->val;
        s.m.b_val = plan->B.full->val;
        if (s.ha.shrunk && cudaMemsetAsync(s.ha.shrunk, 0, sizeof(u32), ctx->stream) != cudaSuccess) rc = spb_fail(SPB_ERR_CUDA, "memset failed");
        s.t_sym = tm.mark();
        if (!rc) rc = mm_numeric(ctx, ws, s, r, mst, tm, s.t_sym);
    } else if (!rc) {
        // fallback: the operands spb_multiply_mm's consolidations return -- the non-empty runs -- through the whole multiply
        spb_coo *Ac = nullptr, *Bc = nullptr;
        spb_coo Aview;
        const spb_coo *Ause = plan->A.full, *Buse = plan->B.full;
        if (plan->A.mode == PO_AS_GIVEN) {
            Aview = *plan->A.full;   // shares the plan's copy of the indices and its cached row structure
            Aview.val = const_cast<double *>(da);
            Aview.owned = false;
            Ause = &Aview;
        } else if (h[0]) {
            rc = pattern_compact(ctx, ws, plan->A, plan->A.runs - h[0], &Ac);
            Ause = Ac;
        }
        if (!rc && h[2]) {
            rc = pattern_compact(ctx, ws, plan->B, plan->B.runs - h[2], &Bc);
            Buse = Bc;
        }
        if (!rc && Ause->n && Buse->n)
            rc = multiply_core(ctx, plan->C, plan->si, Ause, plan->a_row_dim, plan->sj, Buse, plan->b_inner_dim, plan->sk, r, mst, tm, t2);
        spb_coo_free(ctx, Ac);
        spb_coo_free(ctx, Bc);
    }
    if (rc) { spb_coo_free(ctx, r); return rc; }
    *out = r;
    return SPB_OK;
}

}  // extern "C"

// ---- multiply in row panels ------------------------------------------------------------------------------------------
// The A-row loop of spsparse::multiply carries no state from one row to the next (multiply_sparse.hpp:192-246), so the
// product can be formed panel by panel -- a panel is a contiguous range of the non-empty rows of op(A) -- and the panels'
// results, concatenated in panel order, are the reference's output.  This is how products with more than 2^31 entries
// (which no VectorCooArray can hold, algorithm.hpp:419) or more bytes than the GPU has are computed: BASELINE config 4.
struct spb_mm_plan {
    spb_ctx *ctx;
    double C;
    const spb_coo *si, *sj, *sk;   // the caller's scale vectors (must outlive the plan)
    spb_coo *Ac, *Bc;              // consolidated operands owned by the plan (nullptr: the caller's array is used as it is)
    const spb_coo *A, *B;          // what the panels multiply
    int a_row_dim, b_inner_dim;
    u64 shape[2];
    u64 products;                  // F of the whole product
    std::vector<u32> row_lo;       // [panels + 1] compressed row numbers
    std::vector<u32> ent_lo;       // [panels + 1] entry offsets into A
    std::vector<u64> prod_lo;      // [panels + 1] product offsets
    std::vector<i32> row_first;    // [panels] row index i of each panel's first row
    std::vector<i32> row_last;     // [panels] ... and of its last row
};

// rb[c] = first compressed row whose first product has number >= c * chunk (c = nchunks: nrows); eb / pb: its first
// entry and the number of that entry's first product; rid[c]: the row index of row rb[c] (and of row rb[c+1]-1 in rid2)
__global__ void k_panel_bounds(const u32 *__restrict__ arow_start, const i32 *__restrict__ arow_id, const u64 *__restrict__ ent_off,
                               u32 nrows, u64 chunk, u32 nchunks, u32 *rb, u32 *eb, u64 *pb) {
    const u32 c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > nchunks) return;
    u32 lo = 0, hi = nrows;
    if (c == nchunks) lo = nrows;
    else {
        const u64 want = (u64)c * chunk;
        while (lo < hi) {
            const u32 mid = lo + (hi - lo) / 2;
            if (ent_off[arow_start[mid]] < want) lo = mid + 1; else hi = mid;
        }
    }
    rb[c] = lo;
    eb[c] = arow_start[lo];
    pb[c] = ent_off[arow_start[lo]];
}
__global__ void k_rebase_u32(const u32 *__restrict__ src, u64 n, u32 base, u32 *dst) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (u64)gridDim.x * blockDim.x) dst[t] = src[t] - base;
}

extern "C" {

int spb_mm_plan_destroy(spb_mm_plan *plan) {
    if (!plan) return SPB_OK;
    spb_coo_free(plan->ctx, plan->Ac);
    spb_coo_free(plan->ctx, plan->Bc);
    delete plan;
    return SPB_OK;
}

int spb_mm_plan_create(spb_ctx *ctx, double C, const spb_coo *si, const spb_coo *A, char tA, const spb_coo *sj,
                       const spb_coo *B, char tB, const spb_coo *sk, int policy, int zero_nan,
                       uint64_t max_products_per_panel, spb_mm_plan **out, uint64_t *n_panels, uint64_t *products) {
    if (!ctx || !A || !B || !out) return spb_fail(SPB_ERR_ARG, "spb_mm_plan_create: null argument");
    if (A->rank != 2 || B->rank != 2) return spb_fail(SPB_ERR_ARG, "A and B must be rank-2 arrays");
    if (policy < 0 || policy > 2) return spb_fail(SPB_ERR_ARG, "unknown duplicate policy %d", policy);
    if (max_products_per_panel == 0) return spb_fail(SPB_ERR_ARG, "max_products_per_panel must be positive");
    CKR(scale_ok(si, "scalei")); CKR(scale_ok(sj, "scalej")); CKR(scale_ok(sk, "scalek"));
    CK(cudaSetDevice(ctx->device));
    const int a_so[2] = {tA == 'T' ? 1 : 0, tA == 'T' ? 0 : 1};   // multiply_sparse.hpp:167-169
    const int b_so[2] = {tB == 'T' ? 0 : 1, tB == 'T' ? 1 : 0};
    const int b_mine[2] = {b_so[1], b_so[0]};
    if (A->shape[a_so[1]] != B->shape[b_so[1]])  // :172-174
        return spb_fail(SPB_ERR_INNER_DIM, "Inner dimensions for A (%ld) and B (%ld) must match!",
                        (long)A->shape[a_so[1]], (long)B->shape[b_so[1]]);
    spb_mm_plan *p = new spb_mm_plan();
    p->ctx = ctx; p->C = C; p->si = si; p->sj = sj; p->sk = sk; p->Ac = p->Bc = nullptr; p->A = A; p->B = B;
    p->a_row_dim = a_so[0]; p->b_inner_dim = b_mine[0];
    p->shape[0] = A->shape[a_so[0]]; p->shape[1] = B->shape[b_so[0]];
    p->products = 0;
    *out = p;
    if (n_panels) *n_panels = 0;
    if (products) *products = 0;
    // :178-184: the empty product has no panels
    if (C == 0.0 || (si && si->n == 0) || A->n == 0 || (sj && sj->n == 0) || B->n == 0 || (sk && sk->n == 0)) return SPB_OK;
    int rc = 0;
    if (!(A->sort_order[0] == a_so[0] && A->sort_order[1] == a_so[1])) {
        rc = consolidate_core(ctx, A, a_so, a_so, policy, true, zero_nan, &p->Ac, nullptr);
        p->A = p->Ac;
    }
    if (!rc) {
        if (B->sort_order[0] == b_so[0] && B->sort_order[1] == b_so[1])
            rc = consolidate_core(ctx, B, b_mine, b_so, POLICY_KEEP_ALL, false, 0, &p->Bc, nullptr);
        else
            rc = consolidate_core(ctx, B, b_mine, b_so, policy, true, zero_nan, &p->Bc, nullptr);
        p->B = p->Bc;
    }
    if (rc) { spb_mm_plan_destroy(p); *out = nullptr; return rc; }
    if (p->A->n == 0 || p->B->n == 0) return SPB_OK;
    // products per entry of A -> where the panels are cut
    auto body = [&]() -> int {
        Scratch ws(ctx);
        MMOperands m;
        memset(&m, 0, sizeof m);
        m.a_j = p->A->idx[1 - p->a_row_dim]; m.a_val = p->A->val; m.nnz_a = (u32)p->A->n;
        RowIndex ri;
        CKR(build_row_index(ctx, p->A, &ri));
        m.arow_id = ri.id; m.arow_start = ri.start; m.nrows = ri.nrows;
        u32 *bptr;
        CKR(build_dense_ptr(ctx, p->B, p->A->shape[1 - p->a_row_dim], &bptr));
        m.bptr = bptr;
        double *d;
        unsigned char *mask;
        u32 *bad_vec;
        CKR(ws.zeroed(&bad_vec, 1));
        if (si) { CKR(densify(ctx, ws, si, p->shape[0], &d, nullptr, bad_vec)); m.si = d; }
        if (sj) { CKR(densify(ctx, ws, sj, p->A->shape[1 - p->a_row_dim], &d, &mask, bad_vec)); m.sj = d; m.sj_mask = mask; }
        u32 *ent_f;
        u64 *ent_off;
        CKR(ws.get(&ent_f, m.nnz_a));
        CKR(ws.get(&ent_off, (u64)m.nnz_a + 1));
        const u32 cap = (u32)ctx->sm_count * 32;
        ++ctx->launches, k_entry_products<<<grid_for(m.nnz_a, 256, cap), 256, 0, ctx->stream>>>(m, p->A->idx[p->a_row_dim], ent_f);
        CKR((exclusive_scan<u32, u64>(ctx, ws, ent_f, ent_off, m.nnz_a)));
        u64 F = 0;
        u32 h_bad = 0;
        CK(cudaMemcpyAsync(&F, ent_off + m.nnz_a, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(&h_bad, bad_vec, sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
        spb_coo *Am = const_cast<spb_coo *>(p->A);
        u32 *mx = nullptr;
        if (!Am->max_row_len) {
            CKR(ws.zeroed(&mx, 1));
            ++ctx->launches, k_row_maxlen<<<grid_for(ri.nrows, 256, cap), 256, 0, ctx->stream>>>(ri.start, ri.nrows, mx);
            CK(cudaMemcpyAsync(&Am->max_row_len, mx, sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
        }
        CK(cudaStreamSynchronize(ctx->stream));
        if (h_bad) return bad_scale_vector();
        p->products = F;
        u64 nch64 = div_up(F ? F : 1, max_products_per_panel);
        if (nch64 > ri.nrows) nch64 = ri.nrows;   // a panel holds at least one row
        const u32 nch = (u32)nch64;
        const u64 chunk = div_up(F ? F : 1, (u64)nch);  // even panels
        u32 *rb, *eb;
        u64 *pb;
        CKR(ws.get(&rb, (u64)nch + 1)); CKR(ws.get(&eb, (u64)nch + 1)); CKR(ws.get(&pb, (u64)nch + 1));
        ++ctx->launches, k_panel_bounds<<<(u32)div_up((u64)nch + 1, 128), 128, 0, ctx->stream>>>(ri.start, ri.id, ent_off, ri.nrows, chunk, nch, rb, eb, pb);
        CK(cudaGetLastError());
        std::vector<u32> h_rb(nch + 1), h_eb(nch + 1);
        std::vector<u64> h_pb(nch + 1);
        CK(cudaMemcpyAsync(h_rb.data(), rb, (nch + 1) * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(h_eb.data(), eb, (nch + 1) * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(h_pb.data(), pb, (nch + 1) * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        h_rb[0] = 0; h_eb[0] = 0; h_pb[0] = 0;          // rows without products in front of the first cut belong to panel 0
        h_pb[nch] = F;
        for (u32 c = 0; c <= nch; ++c) {               // drop empty panels (a hub row can span several chunks)
            if (c > 0 && c < nch && h_rb[c] == p->row_lo.back()) continue;
            if (c == nch && !p->row_lo.empty() && h_rb[c] == p->row_lo.back()) { p->prod_lo.back() = F; break; }
            p->row_lo.push_back(h_rb[c]); p->ent_lo.push_back(h_eb[c]); p->prod_lo.push_back(h_pb[c]);
        }
        const size_t np = p->row_lo.size() - 1;
        // first / last row index of every panel (information for the caller: which rows of C a panel holds)
        p->row_first.resize(np); p->row_last.resize(np);
        for (size_t c = 0; c < np; ++c) {
            CK(cudaMemcpyAsync(&p->row_first[c], ri.id + p->row_lo[c], sizeof(i32), cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaMemcpyAsync(&p->row_last[c], ri.id + p->row_lo[c + 1] - 1, sizeof(i32), cudaMemcpyDeviceToHost, ctx->stream));
        }
        CK(cudaStreamSynchronize(ctx->stream));
        return 0;
    };
    rc = body();
    if (rc) { spb_mm_plan_destroy(p); *out = nullptr; return rc; }
    if (n_panels) *n_panels = p->row_lo.empty() ? 0 : p->row_lo.size() - 1;
    if (products) *products = p->products;
    return SPB_OK;
}

int spb_mm_plan_info(const spb_mm_plan *plan, uint64_t panel, int32_t *first_row, int32_t *last_row, uint64_t *products,
                     uint64_t *shape) {
    if (!plan) return spb_fail(SPB_ERR_ARG, "spb_mm_plan_info: null plan");
    if (shape) { shape[0] = plan->shape[0]; shape[1] = plan->shape[1]; }
    const size_t np = plan->row_lo.empty() ? 0 : plan->row_lo.size() - 1;
    if (panel >= np) {
        if (first_row || last_row || products) return spb_fail(SPB_ERR_ARG, "panel %llu of %zu", (ull)panel, np);
        return SPB_OK;
    }
    if (first_row) *first_row = plan->row_first[panel];
    if (last_row) *last_row = plan->row_last[panel];
    if (products) *products = plan->prod_lo[panel + 1] - plan->prod_lo[panel];
    return SPB_OK;
}

// one panel: symbolic_only = counts, no result array
static int plan_run(spb_mm_plan *plan, uint64_t panel, bool symbolic_only, spb_coo **out, spb_mm_stats *stats) {
    if (!plan || (!symbolic_only && !out)) return spb_fail(SPB_ERR_ARG, "spb_mm_plan: null argument");
    const size_t np = plan->row_lo.empty() ? 0 : plan->row_lo.size() - 1;
    if (panel >= np) return spb_fail(SPB_ERR_ARG, "panel %llu of %zu", (ull)panel, np);
    spb_ctx *ctx = plan->ctx;
    CK(cudaSetDevice(ctx->device));
    if (stats) memset(stats, 0, sizeof *stats);
    const u32 r0 = plan->row_lo[panel], r1 = plan->row_lo[panel + 1], e0 = plan->ent_lo[panel], e1 = plan->ent_lo[panel + 1];
    // the panel as an operand of its own: rows r0..r1 of op(A), row starts re-based to its first entry
    Scratch ws(ctx);
    u32 *rs;
    CKR(ws.get(&rs, (u64)(r1 - r0) + 1));
    ++ctx->launches, k_rebase_u32<<<grid_for((u64)(r1 - r0) + 1, 256, (u32)ctx->sm_count * 8), 256, 0, ctx->stream>>>(plan->A->row_start + r0, (u64)(r1 - r0) + 1, e0, rs);
    CK(cudaGetLastError());
    spb_coo v = *plan->A;
    v.owned = false;
    v.idx[0] += e0; v.idx[1] += e0; v.val += e0;
    v.n = e1 - e0;
    v.row_start = rs; v.row_id = plan->A->row_id + r0; v.nrows = r1 - r0; v.rows_valid = true;
    v.dense_ptr = nullptr; v.range_ptr = nullptr;
    spb_coo *r = nullptr;
    if (!symbolic_only) {
        CKR(coo_new(ctx, 2, plan->shape, 0, false, &r));
        r->owned = true;
    }
    spb_coo dummy;
    memset(&dummy, 0, sizeof dummy);
    Timer tm(ctx->stream);
    const int t0 = tm.mark();
    int rc = multiply_core(ctx, plan->C, plan->si, &v, plan->a_row_dim, plan->sj, plan->B, plan->b_inner_dim, plan->sk,
                           symbolic_only ? &dummy : r, stats, tm, t0, symbolic_only);
    if (rc) { spb_coo_free(ctx, r); return rc; }
    if (out) *out = r;
    return SPB_OK;
}

int spb_mm_plan_symbolic(spb_mm_plan *plan, uint64_t panel, spb_mm_stats *stats) {
    return plan_run(plan, panel, true, nullptr, stats);
}

int spb_mm_plan_panel(spb_mm_plan *plan, uint64_t panel, spb_coo **out, spb_mm_stats *stats) {
    return plan_run(plan, panel, false, out, stats);
}

}  // extern "C"

extern "C" {

// ---- generators ------------------------------------------------------------------------------------
int spb_gen_dup_coo(spb_ctx *ctx, uint64_t seed, uint64_t i0, uint64_t n, uint64_t ubase, int bits,
                    uint64_t zero_every, spb_coo **out) {
    if (!ctx || !out || bits < 1 || bits > 31 || ubase == 0) return spb_fail(SPB_ERR_ARG, "spb_gen_dup_coo: bad argument");
    const u64 shape[2] = {1ull << bits, 1ull << bits};
    CKR(coo_new(ctx, 2, shape, n, true, out));
    if (n) ++ctx->launches, k_gen_dup_coo<<<grid_for(n, 256, 1u << 20), 256, 0, ctx->stream>>>(seed, i0, n, ubase, bits, zero_every, (*out)->idx[0], (*out)->idx[1], (*out)->val);
    CK(cudaGetLastError());
    return SPB_OK;
}

int spb_gen_banded(spb_ctx *ctx, uint64_t seed, uint64_t mdim, uint64_t r0, uint64_t r1, spb_coo **out) {
    if (!ctx || !out || r1 < r0 || r1 > mdim) return spb_fail(SPB_ERR_ARG, "spb_gen_banded: bad argument");
    const u64 shape[2] = {mdim, mdim};
    const u64 n = (r1 - r0) * 5;
    CKR(coo_new(ctx, 2, shape, n, true, out));
    if (n) ++ctx->launches, k_gen_banded<<<grid_for(n, 256, 1u << 20), 256, 0, ctx->stream>>>(seed, mdim, r0, n, (*out)->idx[0], (*out)->idx[1], (*out)->val);
    CK(cudaGetLastError());
    return SPB_OK;
}

int spb_gen_regrid(spb_ctx *ctx, uint64_t seed, uint32_t ny, uint32_t nx, uint32_t gy, uint32_t gx, spb_coo **out) {
    if (!ctx || !out || !ny || !nx || !gy || !gx) return spb_fail(SPB_ERR_ARG, "spb_gen_regrid: bad argument");
    const u64 shape[2] = {(u64)ny * nx, (u64)gy * gx};
    const u64 n = shape[0] * 4;
    CKR(coo_new(ctx, 2, shape, n, true, out));
    ++ctx->launches, k_gen_regrid<<<grid_for(n, 256, 1u << 20), 256, 0, ctx->stream>>>(seed, ny, nx, gy, gx, n, (*out)->idx[0], (*out)->idx[1], (*out)->val);
    CK(cudaGetLastError());
    return SPB_OK;
}

int spb_gen_rmat(spb_ctx *ctx, uint64_t seed, int scale, uint64_t nedges, spb_coo **out) {
    if (!ctx || !out || scale < 1 || scale > 30) return spb_fail(SPB_ERR_ARG, "spb_gen_rmat: bad argument");
    const u64 shape[2] = {1ull << scale, 1ull << scale};
    CKR(coo_new(ctx, 2, shape, nedges, true, out));
    if (nedges) ++ctx->launches, k_gen_rmat<<<grid_for(nedges, 256, 1u << 20), 256, 0, ctx->stream>>>(seed, scale, nedges, (*out)->idx[0], (*out)->idx[1], (*out)->val);
    CK(cudaGetLastError());
    return SPB_OK;
}

int spb_gen_vector(spb_ctx *ctx, uint64_t seed, uint64_t dim, spb_coo **out) {
    if (!ctx || !out) return spb_fail(SPB_ERR_ARG, "spb_gen_vector: bad argument");
    const u64 shape[1] = {dim};
    CKR(coo_new(ctx, 1, shape, dim, true, out));
    if (dim) ++ctx->launches, k_gen_vector<<<grid_for(dim, 256, 1u << 20), 256, 0, ctx->stream>>>(seed, dim, (*out)->idx[0], (*out)->val);
    CK(cudaGetLastError());
    const int so[1] = {0};
    set_order(*out, so);
    return SPB_OK;
}

}  // extern "C"

// ==================================================================================================
// row-partitioned multiply on the GPUs of one node (one process per GPU); device side in rowpart.cuh
// ==================================================================================================
struct spb_rowpart {
    spb_ctx *ctx;
    int rank, n_ranks;
    u64 row_lo[RP_MAX_RANKS + 1];
    u64 m;                       // rows of B = inner dimension
    u64 cap_entries, cap_rows;   // per-rank capacity of the published shard (the same on every rank)
    u64 slack;                   // entries of room before and after the shard (halo rows of the neighbours)
    int mode;                    // 0: halos fetched in place around the own shard; 1: everything copied (sticky once needed)
    size_t off_ptr, off_cols, off_vals, buf_bytes, region_bytes;   // two buffers (ptr, cols, vals) behind the flags: steps alternate
    void *region;                // this rank's exported allocation
    void *peer_base[RP_MAX_RANKS];
    bool attached;
    cudaStream_t side;
    cudaEvent_t ev_main, ev_pub, ev_pull, ev_t[4];
    u64 step;
    u32 *g_ptr;                  // [m + 2] row pointer of the fetched rows, indexed by the absolute row
    i32 *g_cols;
    double *g_vals;
    u64 g_cap;
    u64 *hull, *info;            // device: [2], [4]
    u32 *error;                  // device
    double *sj_dense;            // [m] dense scalej; only the fetched range is rewritten each step
    unsigned char *sj_mask;
};

static size_t rp_align(size_t x) { return (x + 255) & ~(size_t)255; }

static void rp_layout(spb_rowpart *rp) {
    rp->off_ptr = rp_align(RP_FLAG_WORDS * sizeof(u64));
    rp->off_cols = rp->off_ptr + rp_align((rp->cap_rows + 2) * sizeof(u32));
    rp->off_vals = rp->off_cols + rp_align((rp->cap_entries + 2 * rp->slack) * sizeof(i32));
    rp->buf_bytes = rp->off_vals + rp_align((rp->cap_entries + 2 * rp->slack) * sizeof(double)) - rp->off_ptr;
    rp->region_bytes = rp->off_ptr + 2 * rp->buf_bytes;
}

static void rp_args(const spb_rowpart *rp, RpArgs *a) {
    memset(a, 0, sizeof *a);
    a->rank = rp->rank; a->n_ranks = rp->n_ranks; a->step = rp->step; a->error = rp->error;
    for (int g = 0; g <= rp->n_ranks; ++g) a->row_lo[g] = rp->row_lo[g];
    // Two shard buffers, used by alternate steps: step s is written while the peers may still be reading step s - 1, so a
    // rank only ever waits for the readers of step s - 2 (in practice never) before it consolidates its next shard.
    const size_t par = (size_t)(rp->step & 1) * rp->buf_bytes;
    for (int g = 0; g < rp->n_ranks; ++g) {
        char *b = (char *)rp->peer_base[g];
        a->reg[g].flags = (u64 *)b;
        a->reg[g].ptr = (u32 *)(b + par + rp->off_ptr);
        a->reg[g].cols = (i32 *)(b + par + rp->off_cols) + rp->slack;     // the shard itself; the slack lies on either side
        a->reg[g].vals = (double *)(b + par + rp->off_vals) + rp->slack;
    }
    a->slack = (u32)rp->slack;
}

extern "C" {

int spb_rowpart_destroy(spb_rowpart *rp) {
    if (!rp) return SPB_OK;
    cudaSetDevice(rp->ctx->device);
    cudaStreamSynchronize(rp->ctx->stream);
    if (rp->side) cudaStreamSynchronize(rp->side);
    for (int g = 0; g < rp->n_ranks; ++g)
        if (rp->attached && g != rp->rank && rp->peer_base[g]) cudaIpcCloseMemHandle(rp->peer_base[g]);
    cudaFree(rp->region);
    cudaFree(rp->g_ptr); cudaFree(rp->g_cols); cudaFree(rp->g_vals);
    cudaFree(rp->hull); cudaFree(rp->sj_dense); cudaFree(rp->sj_mask);
    if (rp->side) cudaStreamDestroy(rp->side);
    for (cudaEvent_t e : {rp->ev_main, rp->ev_pub, rp->ev_pull, rp->ev_t[0], rp->ev_t[1], rp->ev_t[2], rp->ev_t[3]})
        if (e) cudaEventDestroy(e);
    delete rp;
    return SPB_OK;
}

int spb_rowpart_create(spb_ctx *ctx, int rank, int n_ranks, const uint64_t *row_lo, uint64_t cap_entries, spb_rowpart **out) {
    if (!ctx || !row_lo || !out) return spb_fail(SPB_ERR_ARG, "spb_rowpart_create: null argument");
    if (n_ranks < 1 || n_ranks > RP_MAX_RANKS || rank < 0 || rank >= n_ranks)
        return spb_fail(SPB_ERR_ARG, "spb_rowpart_create: rank %d of %d (at most %d ranks)", rank, n_ranks, RP_MAX_RANKS);
    for (int g = 0; g < n_ranks; ++g)
        if (row_lo[g] > row_lo[g + 1]) return spb_fail(SPB_ERR_ARG, "spb_rowpart_create: row offsets must not decrease");
    if (row_lo[0] != 0 || row_lo[n_ranks] > (1ull << 31)) return spb_fail(SPB_ERR_ARG, "spb_rowpart_create: bad row offsets");
    if (cap_entries >= (1ull << 31) || cap_entries * (u64)n_ranks >= (1ull << 32))
        return spb_fail(SPB_ERR_TOO_LARGE, "spb_rowpart_create: a shard holds fewer than 2^31 entries, all of B fewer than 2^32");
    CK(cudaSetDevice(ctx->device));
    spb_rowpart *rp = new spb_rowpart();
    memset(rp, 0, sizeof *rp);
    rp->ctx = ctx; rp->rank = rank; rp->n_ranks = n_ranks;
    u64 rows_max = 0;
    for (int g = 0; g <= n_ranks; ++g) rp->row_lo[g] = row_lo[g];
    for (int g = 0; g < n_ranks; ++g) rows_max = std::max<u64>(rows_max, row_lo[g + 1] - row_lo[g]);
    rp->m = row_lo[n_ranks];
    rp->cap_entries = cap_entries ? cap_entries : 1;
    rp->cap_rows = rows_max;
    rp->slack = ((rp->cap_entries / 16 > 4096 ? rp->cap_entries / 16 : 4096) + 63) & ~63ull;   // multiple of 64 entries: alignment kept
    rp->mode = 0;
    rp_layout(rp);
    *out = rp;
    auto body = [&]() -> int {
        if (n_ranks > 1) {
            CK(cudaMalloc(&rp->region, rp->region_bytes));
            CK(cudaMemset(rp->region, 0, rp->region_bytes));   // step counters and pointers start at 0
            rp->g_cap = rp->cap_entries * (u64)n_ranks;   // the copy buffers themselves are allocated when first needed
            CK(cudaMalloc((void **)&rp->g_ptr, (rp->m + 2) * sizeof(u32)));
            CK(cudaMalloc((void **)&rp->hull, 8 * sizeof(u64)));
            CK(cudaMemset(rp->hull, 0, 8 * sizeof(u64)));
            rp->info = rp->hull + 2;
            rp->error = (u32 *)(rp->hull + 6);
            int lo_pri = 0, hi_pri = 0;
            CK(cudaDeviceGetStreamPriorityRange(&lo_pri, &hi_pri));
            // small kernels: ahead of the sort's blocks (SPB_ROWPART_SIDE_PRIO=0: the default priority, for A/B runs)
            const bool side_hi = !(getenv("SPB_ROWPART_SIDE_PRIO") && atoi(getenv("SPB_ROWPART_SIDE_PRIO")) == 0);
            CK(cudaStreamCreateWithPriority(&rp->side, cudaStreamNonBlocking, side_hi ? hi_pri : lo_pri));
            CK(cudaEventCreateWithFlags(&rp->ev_main, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&rp->ev_pub, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&rp->ev_pull, cudaEventDisableTiming));
            for (int i = 0; i < 4; ++i) CK(cudaEventCreate(&rp->ev_t[i]));
        }
        rp->peer_base[rank] = rp->region;
        rp->attached = n_ranks == 1;
        return 0;
    };
    int rc = body();
    if (rc) { spb_rowpart_destroy(rp); *out = nullptr; }
    return rc;
}

int spb_rowpart_handle(spb_rowpart *rp, void *handle, uint64_t handle_bytes) {
    if (!rp || !handle) return spb_fail(SPB_ERR_ARG, "spb_rowpart_handle: null argument");
    if (handle_bytes < sizeof(cudaIpcMemHandle_t)) return spb_fail(SPB_ERR_ARG, "spb_rowpart_handle: %zu bytes needed", sizeof(cudaIpcMemHandle_t));
    memset(handle, 0, handle_bytes);
    if (rp->n_ranks == 1) return SPB_OK;
    CK(cudaSetDevice(rp->ctx->device));
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, rp->region));
    memcpy(handle, &h, sizeof h);
    return SPB_OK;
}

int spb_rowpart_attach(spb_rowpart *rp, const void *handles, uint64_t handle_bytes) {
    if (!rp || !handles) return spb_fail(SPB_ERR_ARG, "spb_rowpart_attach: null argument");
    if (handle_bytes < sizeof(cudaIpcMemHandle_t)) return spb_fail(SPB_ERR_ARG, "spb_rowpart_attach: bad handle size");
    if (rp->attached) return SPB_OK;
    CK(cudaSetDevice(rp->ctx->device));
    for (int g = 0; g < rp->n_ranks; ++g) {
        if (g == rp->rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char *)handles + (size_t)g * handle_bytes, sizeof h);
        void *p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess)
            return spb_fail(SPB_ERR_CUDA, "cannot map the shard buffer of rank %d (cudaIpcOpenMemHandle: %s); the ranks must be "
                            "processes on one node whose GPUs have peer access", g, cudaGetErrorString(e));
        rp->peer_base[g] = p;
    }
    rp->attached = true;
    return SPB_OK;
}

int spb_rowpart_multiply(spb_rowpart *rp, double C, const spb_coo *si, const spb_coo *A, const spb_coo *sj, const spb_coo *B,
                         const spb_coo *sk, int policy, int zero_nan, int fetch_all, spb_coo **out, spb_rowpart_stats *stats) {
    if (!rp || !A || !B || !out) return spb_fail(SPB_ERR_ARG, "spb_rowpart_multiply: null argument");
    if (!rp->attached) return spb_fail(SPB_ERR_ARG, "spb_rowpart_multiply: spb_rowpart_attach has not been called");
    if (A->rank != 2 || B->rank != 2) return spb_fail(SPB_ERR_ARG, "A and B must be rank-2 arrays");
    if (policy < 0 || policy > 2) return spb_fail(SPB_ERR_ARG, "unknown duplicate policy %d", policy);
    CKR(scale_ok(si, "scalei")); CKR(scale_ok(sj, "scalej")); CKR(scale_ok(sk, "scalek"));
    spb_ctx *ctx = rp->ctx;
    CK(cudaSetDevice(ctx->device));
    if (stats) memset(stats, 0, sizeof *stats);
    if (A->shape[1] != B->shape[0])  // multiply_sparse.hpp:172-174
        return spb_fail(SPB_ERR_INNER_DIM, "Inner dimensions for A (%ld) and B (%ld) must match!", (long)A->shape[1], (long)B->shape[0]);
    if (B->shape[0] != rp->m) return spb_fail(SPB_ERR_ARG, "B has %llu rows, the partition was made for %llu", (ull)B->shape[0], (ull)rp->m);
    const int row_major[2] = {0, 1};
    const u64 shape[2] = {A->shape[0], B->shape[1]};
    spb_coo *r = nullptr;
    CKR(coo_new(ctx, 2, shape, 0, false, &r));
    r->owned = true;
    *out = r;
    Timer tm(ctx->stream);
    const int t0 = tm.mark();
    spb_coo *Ac = nullptr, *Bc = nullptr;
    const int rank = rp->rank, n_ranks = rp->n_ranks;
    const u64 r0 = rp->row_lo[rank], r1 = rp->row_lo[rank + 1];
    // Every rank runs every step of the hand-shake, also when its own operands are empty: the peers count on it.
    const bool nothing = C == 0.0 || (si && si->n == 0) || (sj && sj->n == 0) || (sk && sk->n == 0);   // multiply_sparse.hpp:178-184
    auto body = [&]() -> int {
        if (n_ranks == 1) {
            // consolidate by (row, col); operands already consolidated that way are used as they are
            const spb_coo *Buse = B;
            if (!(B->sort_order[0] == 0 && B->sort_order[1] == 1)) {
                CKR(consolidate_core(ctx, B, row_major, row_major, policy, true, zero_nan, &Bc, stats ? &stats->b : nullptr));
                Buse = Bc;
            }
            const int t_b = tm.mark();
            const spb_coo *Ause = A;
            if (!(A->sort_order[0] == 0 && A->sort_order[1] == 1)) {
                CKR(consolidate_core(ctx, A, row_major, row_major, policy, true, zero_nan, &Ac, stats ? &stats->a : nullptr));
                Ause = Ac;
            }
            const int t_a = tm.mark();
            if (!nothing && Ause->n && Buse->n)
                CKR(multiply_core(ctx, C, si, Ause, 0, sj, Buse, 0, sk, r, stats ? &stats->mm : nullptr, tm, t_a));
            if (stats) {
                stats->ms_consolidate_b = tm.ms(t0, t_b); stats->ms_consolidate_a = tm.ms(t_b, t_a);
                stats->rows_fetched = rp->m; stats->entries_fetched = Buse->n;
                const int t_end = tm.mark();
                stats->ms_total = tm.ms(t0, t_end);
            }
            return 0;
        }
        ++rp->step;
        RpArgs ra;
        rp_args(rp, &ra);
        if (B->n > rp->cap_entries)
            return spb_fail(SPB_ERR_TOO_LARGE, "the shard of B has %llu entries, the partition was created for %llu", (ull)B->n, (ull)rp->cap_entries);
        // ---- B shard (main stream): consolidated straight into the buffer the peers read, once they are done with the
        //      previous step's shard; then its row pointers are published and the ready counters raised -------------------------
        CK(cudaMemsetAsync(rp->info, 0, 6 * sizeof(u64), ctx->stream));   // counters of the fetch, error and bad-vector flags
        ++ctx->launches, k_rp_wait_done<<<1, 32, 0, ctx->stream>>>(ra);
        const spb_coo *Buse = B;
        const bool b_sorted = B->sort_order[0] == 0 && B->sort_order[1] == 1;
        if (!b_sorted) {
            CKR(consolidate_core(ctx, B, row_major, row_major, policy, true, zero_nan, &Bc, stats ? &stats->b : nullptr,
                                 ra.reg[rank].cols, ra.reg[rank].vals));
            Buse = Bc;
        }
        const int t_b = tm.mark();
        u32 *local_ptr = nullptr;
        CKR(spb_coo_dense_ptr_range(ctx, Buse, r0, r1, &local_ptr));
        CK(cudaEventRecord(rp->ev_main, ctx->stream));   // A (and B) are complete on the caller's stream from here on
        if (b_sorted) ++ctx->launches, k_rp_publish<<<(u32)ctx->sm_count * 2, 512, 0, ctx->stream>>>(ra, local_ptr, (u32)(r1 - r0), Buse->idx[1], Buse->val);
        else ++ctx->launches, k_rp_publish_ptr<<<(u32)ctx->sm_count, 512, 0, ctx->stream>>>(ra, local_ptr, (u32)(r1 - r0), (u32)Buse->n);
        ++ctx->launches, k_rp_signal_ready<<<1, 32, 0, ctx->stream>>>(ra);
        CK(cudaGetLastError());
        CK(cudaEventRecord(rp->ev_pub, ctx->stream));
        // ---- side stream: hull of A's inner indices, fetch of those rows of B, scalej for that range ---------------------
        const bool copy_mode = fetch_all || rp->mode == 1;
        if (copy_mode && !rp->g_cols) {
            CK(cudaMalloc((void **)&rp->g_cols, rp->g_cap * sizeof(i32)));
            CK(cudaMalloc((void **)&rp->g_vals, rp->g_cap * sizeof(double)));
        }
        CK(cudaStreamWaitEvent(rp->side, rp->ev_main, 0));
        CK(cudaEventRecord(rp->ev_t[0], rp->side));
        if (fetch_all && rp->m) ++ctx->launches, k_rp_hull_set<<<1, 1, 0, rp->side>>>(rp->hull, 0ull, rp->m - 1);
        else {
            ++ctx->launches, k_rp_hull_set<<<1, 1, 0, rp->side>>>(rp->hull, ~0ull, 0ull);   // empty until an entry of A is seen
            if (A->n) ++ctx->launches, k_rp_hull<<<grid_for(A->n, 256, (u32)ctx->sm_count * 4), 256, 0, rp->side>>>(A->idx[1], A->n, rp->hull);
        }
        CK(cudaStreamWaitEvent(rp->side, rp->ev_pub, 0));
        CK(cudaEventRecord(rp->ev_t[1], rp->side));
        ++ctx->launches, k_rp_wait_ready<<<1, 32, 0, rp->side>>>(ra, rp->hull);   // one warp waits for the peers; the fetch's blocks do not
        ++ctx->launches;
        if (copy_mode) k_rp_pull<false><<<96u, RP_PULL_THREADS, 0, rp->side>>>(ra, rp->hull, rp->g_ptr, rp->g_cols, rp->g_vals, rp->g_cap, rp->info);
        else k_rp_pull<true><<<32u, RP_PULL_THREADS, 0, rp->side>>>(ra, rp->hull, rp->g_ptr, nullptr, nullptr, 0, rp->info);
        CK(cudaEventRecord(rp->ev_t[2], rp->side));
        u32 *bad_vec = (u32 *)(rp->hull + 7);
        if (sj) {
            if (!rp->sj_dense) {
                CK(cudaMalloc((void **)&rp->sj_dense, (rp->m ? rp->m : 1) * sizeof(double)));
                CK(cudaMalloc((void **)&rp->sj_mask, rp->m ? rp->m : 1));
            }
            ++ctx->launches, k_rp_zero_range<<<(u32)ctx->sm_count, 512, 0, rp->side>>>(rp->hull, rp->sj_dense, rp->sj_mask);
            if (sj->n) ++ctx->launches, k_rp_densify_range<<<grid_for(sj->n, 256, (u32)ctx->sm_count * 4), 256, 0, rp->side>>>(sj->idx[0], sj->val, sj->n, rp->hull, rp->sj_dense, rp->sj_mask, bad_vec);
        }
        CK(cudaGetLastError());
        CK(cudaEventRecord(rp->ev_t[3], rp->side));
        CK(cudaEventRecord(rp->ev_pull, rp->side));
        // ---- A block (main stream, while the fetch runs) ---------------------------------------------------------------------
        const spb_coo *Ause = A;
        if (!(A->sort_order[0] == 0 && A->sort_order[1] == 1)) {
            CKR(consolidate_core(ctx, A, row_major, row_major, policy, true, zero_nan, &Ac, stats ? &stats->a : nullptr));
            Ause = Ac;
        }
        const int t_a = tm.mark();
        bool in_place = !copy_mode;
        if (in_place) {
            // did the halos fit the slack?  (the fetch is long finished: consolidate(A) ran meanwhile)
            u64 outcome = 0;
            CK(cudaEventSynchronize(rp->ev_pull));
            CK(cudaMemcpyAsync(&outcome, rp->info + 3, sizeof outcome, cudaMemcpyDeviceToHost, rp->side));
            CK(cudaStreamSynchronize(rp->side));
            if (outcome == 3) {
                // no: this block of A reaches far into the neighbours' rows.  Copy everything (now, and from now on).
                rp->mode = 1;
                in_place = false;
                if (!rp->g_cols) {
                    CK(cudaMalloc((void **)&rp->g_cols, rp->g_cap * sizeof(i32)));
                    CK(cudaMalloc((void **)&rp->g_vals, rp->g_cap * sizeof(double)));
                }
                CK(cudaMemsetAsync(rp->info, 0, 4 * sizeof(u64), rp->side));
                ++ctx->launches, k_rp_pull<false><<<96u, RP_PULL_THREADS, 0, rp->side>>>(ra, rp->hull, rp->g_ptr, rp->g_cols, rp->g_vals, rp->g_cap, rp->info);
                CK(cudaGetLastError());
                CK(cudaEventRecord(rp->ev_pull, rp->side));
            }
        }
        CK(cudaStreamWaitEvent(ctx->stream, rp->ev_pull, 0));
        const int t_w = tm.mark();
        // ---- multiply against the fetched rows ----------------------------------------------------------------------------------
        spb_coo Bv;
        memset(&Bv, 0, sizeof Bv);
        Bv.rank = 2; Bv.shape[0] = B->shape[0]; Bv.shape[1] = B->shape[1];
        Bv.n = Buse->n * (u64)n_ranks;          // estimate (kernel-variant heuristics only); the count fetched is in stats
        Bv.idx[0] = nullptr;
        Bv.idx[1] = in_place ? ra.reg[rank].cols - rp->slack : rp->g_cols;   // in place: [lower halo | own shard | upper halo]
        Bv.val = in_place ? ra.reg[rank].vals - rp->slack : rp->g_vals;
        Bv.sort_order[0] = 0; Bv.sort_order[1] = 1;
        Bv.dense_ptr = rp->g_ptr; Bv.dense_ptr_owned = false;
        PreScale pre = {rp->sj_dense, rp->sj_mask};
        if (!nothing && Ause->n)
            CKR(multiply_core(ctx, C, si, Ause, 0, sj, &Bv, 0, sk, r, stats ? &stats->mm : nullptr, tm, t_w, false, sj ? &pre : nullptr));
        u64 h_info[6];
        CK(cudaMemcpyAsync(h_info, rp->info, sizeof h_info, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        const u32 h_err = (u32)h_info[4], h_bad = (u32)(h_info[5]);
        if (h_err == 2) return spb_fail(SPB_ERR_TOO_LARGE, "the rows of B this rank needs hold %llu entries; the partition's buffers hold %llu", (ull)h_info[0], (ull)rp->g_cap);
        if (h_err == 4) return spb_fail(SPB_ERR_ARG, "the shard of B holds entries of rows outside [%llu, %llu): not this rank's rows", (ull)r0, (ull)r1);
        if (h_err) return spb_fail(SPB_ERR_CUDA, "row-partitioned multiply: a peer did not publish its shard of B within %llu s", (ull)(RP_TIMEOUT_NS / 1000000000ull));
        if (sj && h_bad) return bad_scale_vector();
        if (stats) {
            stats->entries_fetched = h_info[0]; stats->rows_fetched = h_info[1];
            stats->mm.nnz_b = h_info[0];
            stats->ms_consolidate_b = tm.ms(t0, t_b); stats->ms_consolidate_a = tm.ms(t_b, t_a); stats->ms_fetch_wait = tm.ms(t_a, t_w);
            float f = 0;
            cudaEventElapsedTime(&f, rp->ev_t[1], rp->ev_t[2]); stats->ms_fetch = f;
            cudaEventElapsedTime(&f, rp->ev_t[0], rp->ev_t[3]); stats->ms_side_stream = f;
            const int t_end = tm.mark();
            stats->ms_total = tm.ms(t0, t_end);
        }
        return 0;
    };
    int rc = body();
    spb_coo_free(ctx, Ac);
    spb_coo_free(ctx, Bc);
    if (rc) { spb_coo_free(ctx, r); *out = nullptr; }
    return rc;
}

}  // extern "C"
