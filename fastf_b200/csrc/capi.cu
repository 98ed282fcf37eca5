// libfastf_gpu.so -- implementation of include/fastf_gpu.h: host orchestration of the sm_100a kernels.
//
// Everything that touches read data runs on the device (kernels in the .cuh files next to this one).
// The host side here only (a) walks the BGZF BSIZE chain (~20 bytes per <= 64 KiB block), (b) moves
// bytes, (c) sizes buffers from device-side counters and (d) launches.  There is no CPU fallback:
// without a CUDA device fastf_ctx_create fails and nothing else can be called.
//
// Streams: `compute` runs the per-chunk chain  header? -> inflate -> parse -> counts -> gather;
// `copy` brings the next chunk's compressed bytes in (fastf_bam2db_feed) while the previous chunk is
// inflating; `mt` extends the MT19937 keep-bit stream while chunks are being parsed.  Per-chunk state
// is double buffered ("slots"), so the only host wait per chunk is for the previous chunk's 32-byte
// counter snapshot, which sizes the candidate array.
//
// One translation unit in six files: this one holds the context, the allocation caches, the D2H helper and the sampling
// contract; capi_launch.cuh (engines, string tables, block index), capi_bam2db.cuh (the job), capi_blocks.cuh (building blocks for
// multi-GPU hosts, single-kernel wrappers), capi_freq.cuh and capi_taghist.cuh are included at the end, in that order.  The
// one-process multi-GPU driver is a separate unit on top of the public C-ABI (sharded.cu).
//
// Resources free themselves: a DevBuf / PinBuf gives its allocation back to the context's pool when it is destroyed, an Event destroys
// its CUDA event, and the structs made of them (the job, its chunk slots, the scratch sets) need no release code.  A function that owns
// buffers declares a DrainOnExit after them, so that none goes back to a pool while queued work can still touch it.
#include "../../include/fastf_gpu.h"
#include "common.cuh"
#include "bgzf_index.h"
#include "bgzf_inflate.cuh"
#include "bgzf_inflate_tps.cuh"
#include "bgzf_crc32.cuh"
#include "bam_parse.cuh"
#include "scan_mt_sample.cuh"
#include "radix_dedup.cuh"
#include "mt_jump.h"
#include "freq.cuh"
#include "bam_tags.cuh"
#include "bam_straddle.cuh"
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <thread>
#include <vector>
#include <unordered_map>
#include <string>
#include <chrono>
#ifndef FASTF_EMU
#include <cuda.h>   // driver API: cuMemBatchDecompressAsync (Blackwell hardware decompression engine)
#endif
static double wall_seconds() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

#define FASTF_ABI_VERSION 1

struct PoolEntry { void *p; size_t cap; };
struct fastf_ctx {
    int device;
    cudaStream_t compute, copy, mt, infl;
    char err[1024];
    u32 launches;   // kernels launched through this context (bench: gpu_launches)
    int n_sm;
    bool tps_attr_set;
    bool crc_attr_set;
    u64 taghist_chunk_blocks = 0, taghist_round0_mask = 0;   // fastf_taghist_test_hooks
    void *mtj_polys;   // device copy of x^(2^k) mod phi, k = 0..44 (uploaded on first use)
    // size-bucketed caches of device / pinned allocations: a job's buffers are recycled by the next job on the same
    // context, so steady-state calls do not pay cudaMalloc / cudaMallocHost (both synchronise the device)
    std::vector<PoolEntry> *dev_pool, *pin_pool;
    // Sizes the buffers of the last bam2db job ended with.  A buffer that grows in mid-job drains every stream (dev_reserve) and
    // leaves the device idle while the host queues the next chunk, so the next job starts its growing buffers at these sizes.
    size_t hint_cand = 0, hint_ring = 0;
};

static int ctx_fail(fastf_ctx *ctx, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    if (ctx) vsnprintf(ctx->err, sizeof ctx->err, fmt, ap);
    va_end(ap);
    if (ctx && getenv("FASTF_VERBOSE")) fprintf(stderr, "fastf_gpu: %s\n", ctx->err);
    return 1;
}
#define CK(call)                                                                                                               \
    do {                                                                                                                       \
        cudaError_t e_ = (call);                                                                                               \
        if (e_ != cudaSuccess) return ctx_fail(ctx, "%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));     \
    } while (0)
#define CKL(name)                                                                                                              \
    do {                                                                                                                       \
        ctx->launches++;                                                                                                       \
        cudaError_t e_ = cudaGetLastError();                                                                                   \
        if (e_ != cudaSuccess) return ctx_fail(ctx, "%s:%d: launch of %s -> %s", __FILE__, __LINE__, name, cudaGetErrorString(e_)); \
    } while (0)
#define TRY(expr)                                                                                                              \
    do {                                                                                                                       \
        int r_ = (expr);                                                                                                       \
        if (r_) return r_;                                                                                                     \
    } while (0)

static const char *status_string(u32 st, char *buf, size_t n)
{
    static const char *names[] = {"bad-btype", "bad-stored", "bad-codelens", "bad-symbol", "bad-distance", "out-overflow", "size-mismatch", "in-overrun",
                                  "record-straddles-bgzf-block", "record-corrupt", "umi-too-long", "aux-corrupt", "bad-bam-header", "bgzf-crc32-mismatch", "tag-not-a-string"};
    buf[0] = 0;
    for (u32 b = 0; b < 15; b++)
        if (st & (1u << b)) { strncat(buf, names[b], n - strlen(buf) - 2); strncat(buf, " ", n - strlen(buf) - 1); }
    return buf;
}

// ---- growable device / pinned buffers, recycled through the context's pools ------------------------
static void *pool_take(std::vector<PoolEntry> &pool, size_t bytes)
{
    int best = -1;
    for (size_t i = 0; i < pool.size(); i++)
        if (pool[i].cap >= bytes && (best < 0 || pool[i].cap < pool[(size_t)best].cap)) best = (int)i;
    if (best < 0 || pool[(size_t)best].cap > 2 * bytes + (1u << 20)) return nullptr;   // do not burn a huge buffer on a small request
    void *p = pool[(size_t)best].p;
    pool.erase(pool.begin() + best);
    return p;
}
static size_t pool_cap_of(const std::vector<PoolEntry> &pool, size_t bytes)
{
    size_t best = 0;
    for (auto &e : pool)
        if (e.cap >= bytes && (!best || e.cap < best)) best = e.cap;
    return best;
}
// A device (DevBuf) or pinned (PinBuf) buffer that goes back to the pool of the context it was reserved on when it is destroyed or
// released.  Move-only, so that exactly one owner gives it back.
template <std::vector<PoolEntry> *fastf_ctx::*Pool> struct PoolBuf {
    fastf_ctx *ctx = nullptr;   // set by the first dev_reserve / pin_reserve
    void *p = nullptr;
    size_t cap = 0;
    PoolBuf() = default;
    PoolBuf(const PoolBuf &) = delete;
    PoolBuf &operator=(const PoolBuf &) = delete;
    PoolBuf(PoolBuf &&o) noexcept : ctx(o.ctx), p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    PoolBuf &operator=(PoolBuf &&o) noexcept
    {
        if (this != &o) { release(); ctx = o.ctx; p = o.p; cap = o.cap; o.p = nullptr; o.cap = 0; }
        return *this;
    }
    ~PoolBuf() { release(); }
    void release()
    {
        if (p) (ctx->*Pool)->push_back(PoolEntry{p, cap});
        p = nullptr;
        cap = 0;
    }
    template <class T> T *as() const { return (T *)p; }
};
using DevBuf = PoolBuf<&fastf_ctx::dev_pool>;
using PinBuf = PoolBuf<&fastf_ctx::pin_pool>;

struct DrainOnExit {   // declared after a function's buffers, so that it drains the streams before any of them goes back to the pool
    fastf_ctx *ctx;
    ~DrainOnExit() { cudaStreamSynchronize(ctx->compute); cudaStreamSynchronize(ctx->copy); cudaStreamSynchronize(ctx->infl); cudaStreamSynchronize(ctx->mt); }
};

struct Event {   // a CUDA event, destroyed with its holder (the driver frees a recorded event once its work has completed)
    cudaEvent_t e = nullptr;
    Event() = default;
    Event(const Event &) = delete;
    Event &operator=(const Event &) = delete;
    Event(Event &&o) noexcept : e(o.e) { o.e = nullptr; }
    Event &operator=(Event &&o) noexcept
    {
        if (this != &o) { if (e) cudaEventDestroy(e); e = o.e; o.e = nullptr; }
        return *this;
    }
    ~Event() { if (e) cudaEventDestroy(e); }
    cudaError_t create(unsigned flags = 0) { return cudaEventCreateWithFlags(&e, flags); }   // 0: cudaEventDefault, with timing
    operator cudaEvent_t() const { return e; }
};

static int dev_reserve(fastf_ctx *ctx, DevBuf &b, size_t bytes, size_t keep_bytes = 0, cudaStream_t s = 0)
{
    if (bytes <= b.cap) return 0;
    size_t ncap = std::max(bytes, b.cap + b.cap / 2);
    ncap = (ncap + 255) & ~(size_t)255;
    size_t pc = pool_cap_of(*ctx->dev_pool, ncap);
    void *np = nullptr;
    if (pc && pc <= 2 * ncap + (1u << 20)) { np = pool_take(*ctx->dev_pool, ncap); ncap = pc; }
    if (!np) CK(cudaMalloc(&np, ncap));
    if (b.p) {
        if (keep_bytes) CK(cudaMemcpyAsync(np, b.p, keep_bytes, cudaMemcpyDeviceToDevice, s));
        // the old buffer goes back to the pool: nothing in flight on any of our streams may still touch it
        CK(cudaStreamSynchronize(ctx->compute));
        CK(cudaStreamSynchronize(ctx->copy));
        CK(cudaStreamSynchronize(ctx->infl));
        CK(cudaStreamSynchronize(ctx->mt));
        b.release();
    }
    b.ctx = ctx;
    b.p = np;
    b.cap = ncap;
    return 0;
}
static int pin_reserve(fastf_ctx *ctx, PinBuf &b, size_t bytes)
{
    if (bytes <= b.cap) return 0;
    size_t ncap = std::max(bytes, b.cap * 2);
    ncap = (ncap + 63) & ~(size_t)63;
    if (b.p) {
        CK(cudaStreamSynchronize(ctx->compute));
        CK(cudaStreamSynchronize(ctx->copy));
        CK(cudaStreamSynchronize(ctx->infl));
        CK(cudaStreamSynchronize(ctx->mt));
        b.release();
    }
    b.ctx = ctx;
    size_t pc = pool_cap_of(*ctx->pin_pool, ncap);
    if (pc && pc <= 2 * ncap + (1u << 20)) { b.p = pool_take(*ctx->pin_pool, ncap); b.cap = pc; }
    if (!b.p) { CK(cudaMallocHost(&b.p, ncap)); b.cap = ncap; }
    return 0;
}
static void pools_trim(fastf_ctx *ctx)
{
    for (auto &e : *ctx->dev_pool) cudaFree(e.p);
    for (auto &e : *ctx->pin_pool) cudaFreeHost(e.p);
    ctx->dev_pool->clear();
    ctx->pin_pool->clear();
}

// Large results go to pageable host memory the caller owns (malloc'ed result arrays).  A plain cudaMemcpy into pageable memory is
// staged by the driver at a few GB/s; here the bytes cross PCIe into two pinned bounce buffers (from the context's pool) while
// the host copies the previous piece out, so the transfer runs at memcpy speed.  Synchronous: dst is complete on return.
// memcpy of a bounce piece into the caller's (fresh, never touched) pageable memory: page faults and a single core's copy rate
// would otherwise bound the D2H of a few hundred MB of results, so a few threads take a slice each
static void par_memcpy(void *dst, const void *src, size_t n)
{
    const size_t SLICE = (size_t)4 << 20;
    const unsigned hw = std::thread::hardware_concurrency();
    const size_t nt = std::min<size_t>(std::min<size_t>(hw > 1 ? hw / 2 : 1, 8), n / SLICE);
    if (nt < 2) { memcpy(dst, src, n); return; }
    std::vector<std::thread> th;
    const size_t per = ((n + nt - 1) / nt + 4095) & ~(size_t)4095;
    for (size_t t = 1; t < nt; t++) {
        const size_t o = t * per;
        if (o < n) th.emplace_back([=] { memcpy((u8 *)dst + o, (const u8 *)src + o, std::min(per, n - o)); });
    }
    memcpy(dst, src, std::min(per, n));
    for (auto &x : th) x.join();
}
static int d2h_pageable(fastf_ctx *ctx, void *dst, const void *src_dev, size_t bytes, cudaStream_t s)
{
    if (bytes == 0) return 0;
    const size_t PIECE = (size_t)16 << 20;
    if (bytes <= ((size_t)1 << 20)) {
        CK(cudaMemcpyAsync(dst, src_dev, bytes, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        return 0;
    }
    PinBuf bounce[2];
    Event ev[2];
    DrainOnExit drain{ctx};
    for (int k = 0; k < 2; k++) { TRY(pin_reserve(ctx, bounce[k], PIECE)); if (ev[k].create(cudaEventDisableTiming) != cudaSuccess) return ctx_fail(ctx, "d2h: event creation failed"); }
    const size_t n_pieces = (bytes + PIECE - 1) / PIECE;
    for (size_t k = 0; k <= n_pieces; k++) {
        if (k < n_pieces) {
            const size_t o = k * PIECE, m = std::min(PIECE, bytes - o);
            if (cudaMemcpyAsync(bounce[k & 1].p, (const u8 *)src_dev + o, m, cudaMemcpyDeviceToHost, s) != cudaSuccess || cudaEventRecord(ev[k & 1], s) != cudaSuccess) return ctx_fail(ctx, "d2h: copy failed");
        }
        if (k > 0) {
            const size_t o = (k - 1) * PIECE, m = std::min(PIECE, bytes - o);
            if (cudaEventSynchronize(ev[(k - 1) & 1]) != cudaSuccess) return ctx_fail(ctx, "d2h: copy failed");
            par_memcpy((u8 *)dst + o, bounce[(k - 1) & 1].p, m);
        }
    }
    return 0;
}

struct Timer {   // CUDA-event stopwatch on one stream; accumulates into *acc at collect()
    Event a, b;
    bool armed = false;
    int init() { return a.create() != cudaSuccess || b.create() != cudaSuccess; }
    void start(cudaStream_t s) { cudaEventRecord(a, s); }
    void stop(cudaStream_t s) { cudaEventRecord(b, s); armed = true; }
    void collect(float *acc) { if (armed) { float ms = 0; cudaEventSynchronize(b); cudaEventElapsedTime(&ms, a, b); *acc += ms; armed = false; } }
};

// ---------------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------------
extern "C" int fastf_abi_version(void) { return FASTF_ABI_VERSION; }
#ifndef FASTF_SRC_HASH
#define FASTF_SRC_HASH "unknown"
#endif
#define FASTF_STR2(x) #x
#define FASTF_STR(x) FASTF_STR2(x)
#if FASTF_TPS_PROF
// debug builds only (-DFASTF_TPS_PROF=1, scripts/inflate_ab.py): the kernel's role counters, see bgzf_inflate_tps.cuh
extern "C" int fastf_debug_tps_prof(unsigned long long *out32, int reset)
{
    if (out32 && cudaMemcpyFromSymbol(out32, g_fastf_tps_prof, FASTF_TPS_PROF_N * sizeof(unsigned long long)) != cudaSuccess) return 1;
    if (reset) { unsigned long long z[FASTF_TPS_PROF_N] = {0}; if (cudaMemcpyToSymbol(g_fastf_tps_prof, z, sizeof z) != cudaSuccess) return 1; }
    return 0;
}
#endif
extern "C" const char *fastf_build_info(void)
{
    return "streams=" FASTF_STR(FASTF_TPS_STREAMS) " lanes=" FASTF_STR(FASTF_TPS_LANES) " svc=" FASTF_STR(FASTF_TPS_SVC_WARPS) " lbits=" FASTF_STR(FASTF_TPS_LBITS) " dbits=" FASTF_STR(FASTF_TPS_DBITS)
           " ring=" FASTF_STR(FASTF_TPS_RING) " src=" FASTF_SRC_HASH;
}

static char g_create_err[512] = "";

extern "C" int fastf_ctx_create(int device, fastf_ctx **out)
{
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        snprintf(g_create_err, sizeof g_create_err, "no CUDA device (%s); libfastf_gpu has no CPU path", e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
        return 1;
    }
    if (device < 0 || device >= n) { snprintf(g_create_err, sizeof g_create_err, "device %d out of range (0..%d)", device, n - 1); return 1; }
    if (cudaSetDevice(device) != cudaSuccess) { snprintf(g_create_err, sizeof g_create_err, "cudaSetDevice(%d) failed", device); return 1; }
    fastf_ctx *ctx = (fastf_ctx *)calloc(1, sizeof *ctx);
    ctx->device = device;
    if (cudaStreamCreateWithFlags(&ctx->compute, cudaStreamNonBlocking) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->copy, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->mt, cudaStreamNonBlocking) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->infl, cudaStreamNonBlocking) != cudaSuccess) {
        snprintf(g_create_err, sizeof g_create_err, "cudaStreamCreate failed");
        free(ctx);
        return 1;
    }
#ifdef FASTF_EMU
    ctx->n_sm = 2;
#else
    if (cudaDeviceGetAttribute(&ctx->n_sm, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || ctx->n_sm <= 0) ctx->n_sm = 148;
    // LZ77 match sources are short reads at random places of windows that do not fit the L2 together: a miss should fetch one
    // 32-byte sector, not a 64/128-byte neighbourhood (measured in profiles/: DRAM read traffic of the inflate kernel)
    if (const char *g = getenv("FASTF_L2_FETCH")) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)atoi(g));
#endif
    std::thread([] { fastf_mtj::tables(); }).detach();   // GF(2) jump tables (0.2 s of host work) while the first job streams
    ctx->dev_pool = new std::vector<PoolEntry>();
    ctx->pin_pool = new std::vector<PoolEntry>();
    *out = ctx;
    return 0;
}
extern "C" void fastf_ctx_destroy(fastf_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    if (ctx->mtj_polys) cudaFree(ctx->mtj_polys);
    pools_trim(ctx);
    delete ctx->dev_pool;
    delete ctx->pin_pool;
    cudaStreamDestroy(ctx->compute);
    cudaStreamDestroy(ctx->copy);
    cudaStreamDestroy(ctx->mt);
    cudaStreamDestroy(ctx->infl);
    free(ctx);
}
extern "C" const char *fastf_last_error(const fastf_ctx *ctx) { return ctx ? ctx->err : g_create_err; }
extern "C" uint32_t fastf_launch_count(const fastf_ctx *ctx) { return ctx ? ctx->launches : 0; }
extern "C" void *fastf_compute_stream(const fastf_ctx *ctx) { return ctx ? (void *)ctx->compute : nullptr; }
extern "C" int fastf_host_alloc(fastf_ctx *ctx, size_t bytes, void **out) { CK(cudaSetDevice(ctx->device)); CK(cudaMallocHost(out, bytes ? bytes : 1)); return 0; }
extern "C" void fastf_host_free(fastf_ctx *ctx, void *p) { (void)ctx; if (p) cudaFreeHost(p); }
extern "C" int fastf_device_alloc(fastf_ctx *ctx, size_t bytes, void **out) { CK(cudaSetDevice(ctx->device)); CK(cudaMalloc(out, bytes ? bytes : 1)); return 0; }
extern "C" void fastf_device_free(fastf_ctx *ctx, void *p) { (void)ctx; if (p) cudaFree(p); }
extern "C" int fastf_memcpy_h2d(fastf_ctx *ctx, void *d, const void *s, size_t n) { CK(cudaMemcpyAsync(d, s, n, cudaMemcpyHostToDevice, ctx->compute)); CK(cudaStreamSynchronize(ctx->compute)); return 0; }
static int d2h_pageable(fastf_ctx *ctx, void *dst, const void *src_dev, size_t bytes, cudaStream_t s);
extern "C" int fastf_memcpy_d2h(fastf_ctx *ctx, void *d, const void *s, size_t n) { CK(cudaSetDevice(ctx->device)); return d2h_pageable(ctx, d, s, n, ctx->compute); }
extern "C" int fastf_synchronize(fastf_ctx *ctx) { CK(cudaStreamSynchronize(ctx->copy)); CK(cudaStreamSynchronize(ctx->infl)); CK(cudaStreamSynchronize(ctx->mt)); CK(cudaStreamSynchronize(ctx->compute)); return 0; }
extern "C" void fastf_free(void *p) { free(p); }
extern "C" void fastf_ctx_trim(fastf_ctx *ctx) { if (ctx) { cudaSetDevice(ctx->device); cudaDeviceSynchronize(); pools_trim(ctx); } }

// ---------------------------------------------------------------------------------------------------
// host helpers that define the sampling contract
// ---------------------------------------------------------------------------------------------------
// keep <=> genrand_real1() < rate  with genrand_real1() = genrand_int32()*(1.0/4294967295.0)
// (reference src/mt19937ar.c:149-153) and the comparison done in double against the float rate
// (reference src/bam2db_ds.c:385-390).  The product is monotone in u, so the rule is u < T.
extern "C" uint64_t fastf_keep_threshold(float rate_depth)
{
    const double r = (double)rate_depth;
    if (r <= 0.0) return 0;     // every draw is >= rate: nothing is kept.  A NaN rate falls through: `x >= NaN` is false for every draw, the reference
                                // drops nothing, and the search below ends at 2^32 (keep everything)
    uint64_t lo = 0, hi = 4294967296ull;   // smallest u with u*(1/4294967295) >= r, or 2^32 if none
    while (lo < hi) {
        uint64_t mid = (lo + hi) >> 1;
        double x = (double)(uint32_t)mid * (1.0 / 4294967295.0);
        if (x >= r) hi = mid; else lo = mid + 1;
    }
    return lo;
}

namespace {
struct HostMT {   // Matsumoto-Nishimura mt19937ar, restated (reference src/mt19937ar.c:60-73,105-140); only for SampleInt's <= n_cells draws
    u32 mt[624];
    int mti;
    void init(u32 s)
    {
        mt[0] = s;
        for (mti = 1; mti < 624; mti++) mt[mti] = 1812433253u * (mt[mti - 1] ^ (mt[mti - 1] >> 30)) + (u32)mti;
    }
    u32 next()
    {
        if (mti >= 624) {
            for (int k = 0; k < 624; k++) {
                u32 y = (mt[k] & 0x80000000u) | (mt[(k + 1) % 624] & 0x7fffffffu);
                mt[k] = mt[(k + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
            }
            mti = 0;
        }
        u32 y = mt[mti++];
        y ^= y >> 11;
        y ^= (y << 7) & 0x9d2c5680u;
        y ^= (y << 15) & 0xefc60000u;
        y ^= y >> 18;
        return y;
    }
};
}   // namespace

// reference src/bam2db_ds.c:240-244 + SampleInt src/utils.c:29-75 (without replacement) + qsort(vsI)
extern "C" uint64_t fastf_sample_cells(uint64_t n_cells, float rate_cell, uint32_t seed, uint64_t *out, uint64_t *d0)
{
    const float prod = (float)n_cells * rate_cell;   // size_t * float -> float arithmetic
    if (!(prod >= 0.0f) || prod >= 18446744073709551616.0f) return UINT64_MAX;
    const uint64_t ns = (uint64_t)prod;
    if (ns > n_cells) return UINT64_MAX;             // the reference prints a message and exit(1)s
    if (ns == n_cells) {
        for (uint64_t i = 0; i < n_cells; i++) out[i] = i;
        if (d0) *d0 = 0;
        return ns;
    }
    HostMT mt;
    mt.init(seed);
    std::vector<uint64_t> pool(n_cells);
    for (uint64_t i = 0; i < n_cells; i++) pool[i] = i;
    uint64_t ntotal = n_cells;
    for (uint64_t i = 0; i < ns; i++) {
        uint64_t idx = (uint64_t)mt.next() % ntotal;
        out[i] = pool[idx];
        if (idx != ntotal - 1) pool[idx] = pool[ntotal - 1];
        ntotal--;
    }
    std::sort(out, out + ns);
    if (d0) *d0 = ns;
    return ns;
}

// The reference prints its histogram BST in pre-order (src/filter.c:139-148).  The BST built by inserting keys in read order
// (src/filter.c:105-124) is the Cartesian tree of `first` (first-occurrence ordinal) over the keys in ascending byte order:
// the earliest key is the root, smaller keys form its left subtree, larger ones its right subtree, recursively.
// order_out[k] = index (in ascending key order) of the k-th line of whitelist.txt.  O(n), iterative.
extern "C" int fastf_cartesian_preorder(const uint32_t *first, uint64_t n, uint64_t *order_out)
{
    if (n == 0) return 0;
    const int64_t NIL = -1;
    std::vector<int64_t> left(n, NIL), right(n, NIL), stack;
    stack.reserve(64);
    for (uint64_t i = 0; i < n; i++) {
        int64_t last = NIL;
        while (!stack.empty() && first[stack.back()] > first[i]) { last = stack.back(); stack.pop_back(); }
        left[i] = last;
        if (!stack.empty()) right[stack.back()] = (int64_t)i;
        stack.push_back((int64_t)i);
    }
    const int64_t root = stack.front();
    stack.clear();
    stack.push_back(root);
    uint64_t k = 0;
    while (!stack.empty()) {
        int64_t v = stack.back();
        stack.pop_back();
        order_out[k++] = (uint64_t)v;
        if (right[v] != NIL) stack.push_back(right[v]);
        if (left[v] != NIL) stack.push_back(left[v]);
    }
    return k == n ? 0 : 1;
}

extern "C" int64_t fastf_bgzf_index_host(const void *buf, size_t n, uint64_t *in_off, uint32_t *in_len, uint32_t *isize, uint64_t cap, size_t *consumed)
{
    std::vector<FastfBgzfBlock> blocks;
    size_t used = 0;
    int rc = fastf_bgzf_index((const uint8_t *)buf, n, 0, blocks, &used);
    if (consumed) *consumed = used;
    if (rc != FASTF_BGZF_OK && rc != FASTF_BGZF_NEED_MORE) return -1;
    if (blocks.size() > cap) return -2;
    for (size_t i = 0; i < blocks.size(); i++) { in_off[i] = blocks[i].in_off; in_len[i] = blocks[i].in_len; isize[i] = blocks[i].isize; }
    return (int64_t)blocks.size();
}

#include "capi_launch.cuh"
#include "capi_bam2db.cuh"
#include "capi_blocks.cuh"
#include "capi_freq.cuh"
#include "capi_taghist.cuh"
