// Multi-GPU bam2db inside the library (SURVEY.md 8e): ONE host process drives G devices of a node through the C-ABI of
// include/fastf_gpu.h -- one feeder thread and one context per device -- and exchanges the locally deduplicated keys with an NCCL
// all-to-all (grouped ncclSend / ncclRecv over NVLink) partitioned by cell, so that every (cell, gene) group is counted on one GPU.
//
//   1. the BGZF blocks of the file are sharded contiguously, device by device (records do not straddle blocks in htslib files);
//      the BAM header lies in device 0's shard, later shards run "headerless";
//   2. every device inflates + parses its shard; the per-shard counts {records, CB-valid reads} give each shard the global ordinal
//      of its first CB-valid read = its position in the reference's single MT19937 draw sequence (reference src/bam2db_ds.c:385);
//   3. depth sampling on device at stream index d0 + base + local ordinal; the kept rows (table `umi`, read order) are read back
//      shard by shard when the caller wants them;
//   4. local sort + unique, grouped by destination = order-preserving range partition of the cell index
//      (fastf_unique_partition_device); ONE all-to-all of u64 keys;
//   5. local sort + run-length dedup / count per device; the COO pieces concatenate in device order (cells are range partitioned
//      and every piece is (cell, gene)-sorted), which is the single-GPU result and the reference's `mtx` table.
//
// The depth sweep (fastf_bam2db_run_sharded_sweep) runs the same steps for K sorted thresholds: in step 3 every shard samples at all
// rates at once and keeps each distinct key with its smallest rate index, the exchange carries that index beside the key, and in
// step 5 every device counts each rate over the keys it received (fastf_sweep_count_device).  The single rate is the case K = 1.
//
// This translation unit uses nothing but the public C-ABI, the CUDA runtime and NCCL.  NCCL is bound at run time (dlopen of
// libnccl.so.2: a process that already holds an NCCL -- e.g. one that imported torch -- keeps its own copy).  The emulator build
// (tests, no GPU) replaces the collective by host copies; everything else is the same code.
#include "../../include/fastf_gpu.h"
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>
#ifndef FASTF_EMU   // the emulator build needs no CUDA call here: its "device" memory is host memory
#include <cuda_runtime.h>
#include <dlfcn.h>
#endif

namespace {

#ifndef FASTF_EMU
// the few NCCL entry points of the exchange, declared as in nccl.h 2.x (stable C API)
typedef struct ncclComm *ncclComm_t;
typedef int ncclResult_t;      // ncclSuccess = 0
typedef int ncclDataType_t;    // ncclUint64 = 5
struct Nccl {
    ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
    std::string why;
};
Nccl &nccl()
{
    static Nccl N;
    static bool tried = false;
    if (tried) return N;
    tried = true;
    void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) { N.why = std::string("cannot load libnccl.so.2: ") + dlerror(); return N; }
#define FASTF_NCCL_SYM(field, name) *(void **)(&N.field) = dlsym(h, name); if (!N.field) { N.why = std::string("libnccl lacks ") + name; return N; }
    FASTF_NCCL_SYM(CommInitAll, "ncclCommInitAll")
    FASTF_NCCL_SYM(CommDestroy, "ncclCommDestroy")
    FASTF_NCCL_SYM(GroupStart, "ncclGroupStart")
    FASTF_NCCL_SYM(GroupEnd, "ncclGroupEnd")
    FASTF_NCCL_SYM(Send, "ncclSend")
    FASTF_NCCL_SYM(Recv, "ncclRecv")
    FASTF_NCCL_SYM(GetErrorString, "ncclGetErrorString")
#undef FASTF_NCCL_SYM
    N.ok = true;
    return N;
}
#endif

struct Shard {
    int device = 0;
    fastf_ctx *ctx = nullptr;
    fastf_bam2db_job *job = nullptr;
    size_t byte_lo = 0, byte_hi = 0;
    uint64_t n_rec = 0, n_cbv = 0, n_kept = 0;
    uint64_t *kept = nullptr;              // device, owned by the job
    uint64_t *send = nullptr, *recv = nullptr;   // device
    std::vector<uint64_t> part;            // keys for each destination
    uint64_t n_send = 0, n_recv = 0;
    std::vector<uint64_t> rows;            // kept rows of this shard, read order (want_rows)
    fastf_bam2db_result st;                // stage clocks / byte counts of this shard
    // depth sweep: rate index (position among the sorted thresholds) of every kept / sent / received key and of every row
    uint32_t *kept_rate = nullptr;         // device, owned by the job
    uint32_t *send_rate = nullptr, *recv_rate = nullptr;   // device
    std::vector<uint32_t> row_rate;
    std::vector<uint64_t> sampled, valid, nnz;   // per sorted rate
    std::vector<uint32_t *> coo[3];        // per sorted rate: this device's COO piece (host, malloc'ed by the library)
    float ms_sort = 0, ms_count = 0;
    int rc = 0;
    std::string err;
};

void fail(Shard &s, const char *what)
{
    s.rc = 1;
    const char *e = s.ctx ? fastf_last_error(s.ctx) : fastf_last_error(nullptr);
    s.err = std::string(what) + ": " + (e ? e : "?");
}

// every shard does `fn` on its own host thread (the C-ABI calls block on their device)
template <class F> bool for_all(std::vector<Shard> &S, F fn)
{
#ifdef FASTF_EMU
    for (size_t g = 0; g < S.size(); g++) if (!S[g].rc) fn(S[g], g);   // the SIMT emulator runs one kernel at a time
#else
    std::vector<std::thread> th;
    for (size_t g = 1; g < S.size(); g++) th.emplace_back([&, g] { if (!S[g].rc) fn(S[g], g); });
    if (!S[0].rc) fn(S[0], 0);
    for (auto &t : th) t.join();
#endif
    for (auto &s : S) if (s.rc) return false;
    return true;
}

// the shards of one call and the communicators of its exchange; everything is released when the call returns
struct Run {
    std::vector<Shard> S;
#ifndef FASTF_EMU
    std::vector<ncclComm_t> comms;
#endif
    explicit Run(size_t G) : S(G) {}
    ~Run()
    {
        for (auto &s : S) {
            if (s.ctx) {
                if (s.send) fastf_device_free(s.ctx, s.send);
                if (s.recv) fastf_device_free(s.ctx, s.recv);
                if (s.send_rate) fastf_device_free(s.ctx, s.send_rate);
                if (s.recv_rate) fastf_device_free(s.ctx, s.recv_rate);
            }
            for (auto &v : s.coo) for (auto p : v) fastf_free(p);
            if (s.job) fastf_bam2db_job_free(s.job);
            if (s.ctx) fastf_ctx_destroy(s.ctx);
        }
#ifndef FASTF_EMU
        for (auto c : comms) if (c) nccl().CommDestroy(c);
#endif
    }
};

// CUDA-event stopwatch around blocking C-ABI calls on a shard's compute stream (always 0 in the emulator build, which has no clock)
struct DevClock {
#ifndef FASTF_EMU
    cudaEvent_t a = nullptr, b = nullptr;
    cudaStream_t st;
    explicit DevClock(const Shard &s) : st((cudaStream_t)fastf_compute_stream(s.ctx))
    {
        cudaSetDevice(s.device);
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        cudaEventRecord(a, st);
    }
    float stop()
    {
        float ms = 0;
        if (cudaEventRecord(b, st) == cudaSuccess && cudaEventSynchronize(b) == cudaSuccess) cudaEventElapsedTime(&ms, a, b);
        return ms;
    }
    ~DevClock() { cudaEventDestroy(a); cudaEventDestroy(b); }
#else
    explicit DevClock(const Shard &) {}
    float stop() { return 0; }
#endif
};

}   // namespace

static char g_sharded_err[768] = "";
extern "C" const char *fastf_sharded_last_error(void) { return g_sharded_err; }
static std::atomic<uint64_t> g_fastf_sharded_exchanged{0};
extern "C" uint64_t fastf_sharded_exchanged(void) { return g_fastf_sharded_exchanged.load(); }

static void first_error(const std::vector<Shard> &S)
{
    for (auto &s : S) if (s.rc) { snprintf(g_sharded_err, sizeof g_sharded_err, "device %d: %s", s.device, s.err.c_str()); return; }
}

// 1. block index (host) and contiguous block shards
static int shard_blocks(const char *who, const uint8_t *bytes, size_t n_bytes, const int *devices, std::vector<Shard> &S)
{
    const size_t G = S.size();
    std::vector<uint64_t> in_off;
    std::vector<uint32_t> in_len, isz;
    size_t cap = std::max<size_t>(1024, n_bytes / 8192 + 16), used = 0;   // BGZF blocks of BAM files hold ~20 KB; the index grows on demand
    int64_t nbi;
    for (;;) {
        in_off.resize(cap); in_len.resize(cap); isz.resize(cap);
        nbi = fastf_bgzf_index_host(bytes, n_bytes, in_off.data(), in_len.data(), isz.data(), cap, &used);
        if (nbi != -2) break;
        cap *= 4;
    }
    if (nbi < 0 || used != n_bytes) { snprintf(g_sharded_err, sizeof g_sharded_err, "%s: not a whole BGZF file (index stopped at byte %zu of %zu)", who, used, n_bytes); return 1; }
    const size_t nb = (size_t)nbi;
    // a block starts where the previous one's trailer (CRC32 + ISIZE) ends, whatever its extra field holds
    auto block_start = [&](size_t i) -> size_t { return i == 0 ? 0 : (i < nb ? (size_t)(in_off[i - 1] + in_len[i - 1] + 8) : n_bytes); };
    for (size_t g = 0; g < G; g++) {
        const size_t base = nb / G, rem = nb % G;
        const size_t lo = base * g + std::min(g, rem), hi = lo + base + (g < rem ? 1 : 0);
        S[g].device = devices ? devices[g] : (int)g;
        S[g].byte_lo = block_start(lo);
        S[g].byte_hi = block_start(hi);
    }
    return 0;
}

// 2. contexts, jobs, feed (one host thread per device); then every shard's {records, CB-valid reads}
static int open_and_feed(std::vector<Shard> &S, const fastf_bam2db_params *params, const uint8_t *bytes)
{
    const size_t PIECE = (size_t)128 << 20;
    const bool ok = for_all(S, [&](Shard &s, size_t g) {
        if (fastf_ctx_create(s.device, &s.ctx)) { fail(s, "ctx_create"); return; }
        fastf_bam2db_params p = *params;
        p.headerless = g != 0;
        p.want_rows = 0;   // rows are read back from the device below, before the exchange reorders them
        if (fastf_bam2db_begin(s.ctx, &p, &s.job)) { fail(s, "begin"); return; }
        void *pin[2] = {nullptr, nullptr};
        if (fastf_host_alloc(s.ctx, PIECE, &pin[0]) || fastf_host_alloc(s.ctx, PIECE, &pin[1])) { fail(s, "host_alloc"); return; }
        int which = 0;
        for (size_t at = s.byte_lo; at < s.byte_hi && !s.rc; at += PIECE, which ^= 1) {
            const size_t n = std::min(PIECE, s.byte_hi - at);
            memcpy(pin[which], bytes + at, n);   // page cache / caller's buffer -> pinned ring
            if (fastf_bam2db_feed(s.job, pin[which], n)) fail(s, "feed");
        }
        if (!s.rc && fastf_bam2db_counts(s.job, &s.n_rec, &s.n_cbv)) fail(s, "counts");
        fastf_host_free(s.ctx, pin[0]);
        fastf_host_free(s.ctx, pin[1]);
    });
    if (!ok) first_error(S);
    return ok ? 0 : 1;
}

// global draw ordinal of every shard's first CB-valid read
static std::vector<uint64_t> ordinal_bases(const std::vector<Shard> &S)
{
    std::vector<uint64_t> bases(S.size());
    uint64_t base = 0;
    for (size_t g = 0; g < S.size(); g++) { bases[g] = base; base += S[g].n_cbv; }
    return bases;
}

// 4. the all-to-all of the partitioned keys, and with `rates` of their rate indices beside them (same NCCL group)
static int all_to_all(const char *who, Run &X, bool rates)
{
    std::vector<Shard> &S = X.S;
    const int G = (int)S.size();
    for (int g = 0; g < G; g++) {
        Shard &s = S[(size_t)g];
        s.n_recv = 0;
        for (int p = 0; p < G; p++) s.n_recv += S[(size_t)p].part[(size_t)g];
    }
    const bool ok = for_all(S, [&](Shard &s, size_t) {
        void *d = nullptr;
        if (fastf_device_alloc(s.ctx, (size_t)std::max<uint64_t>(s.n_recv, 1) * 8, &d)) { fail(s, "device_alloc"); return; }
        s.recv = (uint64_t *)d;
        if (rates) {
            if (fastf_device_alloc(s.ctx, (size_t)std::max<uint64_t>(s.n_recv, 1) * 4, &d)) { fail(s, "device_alloc"); return; }
            s.recv_rate = (uint32_t *)d;
        }
    });
    if (!ok) { first_error(S); return 1; }
#ifdef FASTF_EMU
    for (int g = 0; g < G; g++) {   // "device" memory is host memory here
        uint64_t ro = 0;
        for (int p = 0; p < G; p++) {
            uint64_t so = 0;
            for (int q = 0; q < g; q++) so += S[(size_t)p].part[(size_t)q];
            const uint64_t c = S[(size_t)p].part[(size_t)g];
            memcpy(S[(size_t)g].recv + ro, S[(size_t)p].send + so, (size_t)c * 8);
            if (rates) memcpy(S[(size_t)g].recv_rate + ro, S[(size_t)p].send_rate + so, (size_t)c * 4);
            ro += c;
        }
    }
#else
    if (G > 1) {
        Nccl &N = nccl();
        if (!N.ok) { snprintf(g_sharded_err, sizeof g_sharded_err, "%s: NCCL unavailable (%s)", who, N.why.c_str()); return 1; }
        X.comms.assign((size_t)G, nullptr);
        std::vector<int> devs((size_t)G);
        for (int g = 0; g < G; g++) devs[(size_t)g] = S[(size_t)g].device;
        ncclResult_t r = N.CommInitAll(X.comms.data(), G, devs.data());
        if (r) { snprintf(g_sharded_err, sizeof g_sharded_err, "%s: ncclCommInitAll: %s", who, N.GetErrorString(r)); return 1; }
        r = N.GroupStart();
        for (int g = 0; g < G && !r; g++) {
            Shard &s = S[(size_t)g];
            cudaStream_t st = (cudaStream_t)fastf_compute_stream(s.ctx);
            ncclComm_t comm = X.comms[(size_t)g];
            uint64_t so = 0, ro = 0;
            for (int p = 0; p < G && !r; p++) {
                const uint64_t cs = s.part[(size_t)p], cr = S[(size_t)p].part[(size_t)g];
                // per pair of peers the receives match the sends in the order posted: keys, then rate indices
                if (cs) r = N.Send(s.send + so, (size_t)cs, 5 /* ncclUint64 */, p, comm, st);
                if (cs && rates && !r) r = N.Send(s.send_rate + so, (size_t)cs, 3 /* ncclUint32 */, p, comm, st);
                if (cr && !r) r = N.Recv(s.recv + ro, (size_t)cr, 5, p, comm, st);
                if (cr && rates && !r) r = N.Recv(s.recv_rate + ro, (size_t)cr, 3, p, comm, st);
                so += cs; ro += cr;
            }
        }
        ncclResult_t r2 = N.GroupEnd();
        if (r || r2) { snprintf(g_sharded_err, sizeof g_sharded_err, "%s: NCCL all-to-all: %s", who, N.GetErrorString(r ? r : r2)); return 1; }
        for (auto &s : S) { cudaSetDevice(s.device); if (fastf_synchronize(s.ctx)) { fail(s, "synchronize after the exchange"); first_error(S); return 1; } }
    } else if (S[0].n_recv) {
        // on the compute stream, which the counting step uses next: a device-to-device cudaMemcpy may return before the copy ends,
        // and the context's streams do not wait for the legacy default stream
        cudaSetDevice(S[0].device);
        cudaStream_t st = (cudaStream_t)fastf_compute_stream(S[0].ctx);
        if (cudaMemcpyAsync(S[0].recv, S[0].send, (size_t)S[0].n_recv * 8, cudaMemcpyDeviceToDevice, st) != cudaSuccess ||
            (rates && cudaMemcpyAsync(S[0].recv_rate, S[0].send_rate, (size_t)S[0].n_recv * 4, cudaMemcpyDeviceToDevice, st) != cudaSuccess)) {
            snprintf(g_sharded_err, sizeof g_sharded_err, "%s: device copy failed", who);
            return 1;
        }
    }
#endif
    uint64_t x = 0;
    for (auto &s : S) x += s.n_send;
    g_fastf_sharded_exchanged = x;
    return 0;
}

// counters, byte counts and stage clocks over the shards (clocks: the slowest device), laid out like fastf_bam2db_finish's
static void merge_stats(const std::vector<Shard> &S, uint32_t bits_cell, uint32_t bits_gene, uint32_t bits_umi, fastf_bam2db_result *res)
{
    for (auto &s : S) {
        res->total += s.n_rec; res->cb_valid += s.n_cbv;
        res->n_blocks += s.st.n_blocks; res->compressed_bytes += s.st.compressed_bytes; res->inflated_bytes += s.st.inflated_bytes;
        res->status |= s.st.status; res->n_launches += s.st.n_launches; res->n_chunks += s.st.n_chunks;
        res->ms_inflate = std::max(res->ms_inflate, s.st.ms_inflate); res->ms_parse = std::max(res->ms_parse, s.st.ms_parse); res->ms_crc = std::max(res->ms_crc, s.st.ms_crc);
        res->ms_mt = std::max(res->ms_mt, s.st.ms_mt); res->ms_sample = std::max(res->ms_sample, s.st.ms_sample); res->ms_device_total = std::max(res->ms_device_total, s.st.ms_device_total);
        res->ms_sort = std::max(res->ms_sort, s.ms_sort); res->ms_count = std::max(res->ms_count, s.ms_count);
    }
    res->bits_cell = bits_cell; res->bits_gene = bits_gene; res->bits_umi = bits_umi; res->umi_max_bytes = (bits_umi - 4) / 8;
}

// Steps 1-6 for K thresholds sorted ascending (`thr`), or with thr null (K = 1) at the keep threshold of `params`.  res->rate[p] is
// sorted rate p; with the sweep's want_rows, row_rate holds the sorted position of every row's rate.  A key's rate index in the
// single-job result is the minimum over all its copies in the file; the minimum is associative, so every shard reduces its own copies
// before the exchange (fastf_unique_partition_rates_device) and the receiving device reduces again over what the senders delivered
// (fastf_sweep_count_device).  The cell-range partition puts every (cell, gene) group on one device, whose group rates are therefore
// computed from complete data.
static int run_shards(const char *who, int n_devices, const int *devices, const fastf_bam2db_params *params, const void *bgzf_bytes, size_t n_bytes, uint32_t K, const uint64_t *thr,
                      fastf_bam2db_sweep_result *res)
{
    g_sharded_err[0] = 0;
    memset(res, 0, sizeof *res);
    if (n_devices < 1 || n_devices > 64) { snprintf(g_sharded_err, sizeof g_sharded_err, "%s: %d devices", who, n_devices); return 1; }
    const bool sweep = thr != nullptr;
    const int G = n_devices;
    const uint8_t *bytes = (const uint8_t *)bgzf_bytes;
    Run X((size_t)G);
    std::vector<Shard> &S = X.S;
    if (shard_blocks(who, bytes, n_bytes, devices, S) || open_and_feed(S, params, bytes)) return 1;

    // ---- 3. global draw ordinals, sampling, rows, local unique + partition (the sweep: with the smallest rate index per key) ----
    uint32_t bits_cell = 0, bits_gene = 0, bits_umi = 0;
    const std::vector<uint64_t> bases = ordinal_bases(S);
    bool ok = for_all(S, [&](Shard &s, size_t g) {
        s.sampled.assign(K, 0);
        s.valid.assign(K, 0);
        if (sweep ? fastf_bam2db_sample_sweep(s.job, bases[g], K, thr, s.sampled.data(), s.valid.data()) || fastf_bam2db_kept_sweep_device(s.job, &s.kept, &s.kept_rate, &s.n_kept)
                  : fastf_bam2db_sample(s.job, bases[g]) || fastf_bam2db_sample_counts(s.job, &s.sampled[0], &s.valid[0]) || fastf_bam2db_kept_device(s.job, &s.kept, &s.n_kept)) {
            fail(s, "sample");
            return;
        }
        uint32_t bc, bg, bu;
        if (fastf_bam2db_key_layout(s.job, &bc, &bg, &bu)) { fail(s, "key_layout"); return; }
        if (g == 0) { bits_cell = bc; bits_gene = bg; bits_umi = bu; }
        if (params->want_rows && s.n_kept) {   // before the partition, which overwrites the kept keys in place
            s.rows.resize((size_t)s.n_kept);
            if (fastf_memcpy_d2h(s.ctx, s.rows.data(), s.kept, (size_t)s.n_kept * 8)) { fail(s, "rows d2h"); return; }
            if (sweep) {
                s.row_rate.resize((size_t)s.n_kept);
                if (fastf_memcpy_d2h(s.ctx, s.row_rate.data(), s.kept_rate, (size_t)s.n_kept * 4)) { fail(s, "rows d2h"); return; }
            }
        }
        void *d = nullptr;
        if (fastf_device_alloc(s.ctx, (size_t)std::max<uint64_t>(s.n_kept, 1) * 8, &d)) { fail(s, "device_alloc"); return; }
        s.send = (uint64_t *)d;
        if (sweep) {
            if (fastf_device_alloc(s.ctx, (size_t)std::max<uint64_t>(s.n_kept, 1) * 4, &d)) { fail(s, "device_alloc"); return; }
            s.send_rate = (uint32_t *)d;
        }
        s.part.assign((size_t)G, 0);
        DevClock clock(s);
        if (sweep ? fastf_unique_partition_rates_device(s.ctx, s.kept, s.kept_rate, s.n_kept, bc + bg + bu, bg, bu, params->n_cells, (uint32_t)G, s.send, s.send_rate, s.part.data())
                  : fastf_unique_partition_device(s.ctx, s.kept, s.n_kept, bc + bg + bu, bg, bu, params->n_cells, (uint32_t)G, s.send, s.part.data())) {
            fail(s, "unique_partition");
            return;
        }
        s.ms_sort = clock.stop();
        s.n_send = 0;
        for (auto c : s.part) s.n_send += c;
    });
    if (!ok) { first_error(S); return 1; }
    const uint32_t key_bits = bits_cell + bits_gene + bits_umi;

    // ---- 4. the all-to-all of the keys (the sweep: with their rate indices) ----
    if (all_to_all(who, X, sweep)) return 1;

    // ---- 5. per device: every rate's COO piece, back on the host ----
    ok = for_all(S, [&](Shard &s, size_t) {
        s.nnz.assign(K, 0);
        for (auto &v : s.coo) v.assign(K, nullptr);
        DevClock clock(s);
        if (sweep ? fastf_sweep_count_device(s.ctx, s.recv, s.recv_rate, s.n_recv, key_bits, bits_gene, bits_umi, K, s.nnz.data(), s.coo[0].data(), s.coo[1].data(), s.coo[2].data())
                  : fastf_sort_u64_device(s.ctx, s.recv, nullptr, s.n_recv, key_bits) ||
                        fastf_dedup_count_device(s.ctx, s.recv, s.n_recv, bits_gene, bits_umi, &s.nnz[0], &s.coo[0][0], &s.coo[1][0], &s.coo[2][0])) {
            fail(s, "count");
            return;
        }
        s.ms_count = clock.stop();
        memset(&s.st, 0, sizeof s.st);
        if (fastf_bam2db_stats(s.job, &s.st)) { fail(s, "stats"); return; }
    });
    if (!ok) { first_error(S); return 1; }

    // ---- 6. the result, laid out like fastf_bam2db_finish_sweep's in sorted rate order ----
    fastf_bam2db_result st;
    memset(&st, 0, sizeof st);
    merge_stats(S, bits_cell, bits_gene, bits_umi, &st);
    bool oom = false;
    for (uint32_t p = 0; p < K && !oom; p++) {
        fastf_bam2db_result &r = res->rate[p];
        r = st;
        for (auto &s : S) { r.sampled += s.sampled[p]; r.valid += s.valid[p]; r.nnz += s.nnz[p]; }
        r.m_gene = (uint32_t *)malloc(std::max<uint64_t>(r.nnz, 1) * 4);
        r.m_cell = (uint32_t *)malloc(std::max<uint64_t>(r.nnz, 1) * 4);
        r.m_count = (uint32_t *)malloc(std::max<uint64_t>(r.nnz, 1) * 4);
        oom = !r.m_gene || !r.m_cell || !r.m_count;
        uint32_t *dst[3] = {r.m_gene, r.m_cell, r.m_count};
        uint64_t o = 0;
        for (auto &s : S) {
            if (oom) break;
            for (int c = 0; c < 3; c++) if (s.nnz[p]) memcpy(dst[c] + o, s.coo[c][p], (size_t)s.nnz[p] * 4);
            o += s.nnz[p];
        }
    }
    if (!oom && params->want_rows) {
        uint64_t n_rows = 0;
        for (auto &s : S) n_rows += s.rows.size();
        res->row_keys = (uint64_t *)malloc(std::max<uint64_t>(n_rows, 1) * 8);
        res->row_rate = sweep ? (uint8_t *)malloc(std::max<uint64_t>(n_rows, 1)) : nullptr;
        oom = !res->row_keys || (sweep && !res->row_rate);
        uint64_t ro = 0;
        for (auto &s : S) {
            if (oom) break;
            memcpy(res->row_keys + ro, s.rows.data(), s.rows.size() * 8);
            for (size_t k = 0; k < s.row_rate.size(); k++) res->row_rate[ro + k] = (uint8_t)s.row_rate[k];
            ro += s.rows.size();
        }
        res->n_rows = oom ? 0 : n_rows;
    }
    if (oom) {
        snprintf(g_sharded_err, sizeof g_sharded_err, "%s: out of host memory", who);
        fastf_bam2db_sweep_result_free(res);
        return 1;
    }
    res->n_rates = K;
    return 0;
}

extern "C" int fastf_bam2db_run_sharded(int n_devices, const int *devices, const fastf_bam2db_params *params, const void *bgzf_bytes, size_t n_bytes, fastf_bam2db_result *res)
{
    memset(res, 0, sizeof *res);
    fastf_bam2db_sweep_result one;
    if (run_shards("run_sharded", n_devices, devices, params, bgzf_bytes, n_bytes, 1, nullptr, &one)) return 1;
    *res = one.rate[0];
    res->row_keys = one.row_keys;
    res->n_rows = one.n_rows;
    return 0;
}

extern "C" int fastf_bam2db_run_sharded_sweep(int n_devices, const int *devices, const fastf_bam2db_params *params, const void *bgzf_bytes, size_t n_bytes, uint32_t n_rates,
                                              const uint64_t *keep_thresholds, fastf_bam2db_sweep_result *res)
{
    const char *who = "run_sharded_sweep";
    g_sharded_err[0] = 0;
    memset(res, 0, sizeof *res);
    if (n_rates < 1 || n_rates > FASTF_SWEEP_MAX_RATES || !keep_thresholds) { snprintf(g_sharded_err, sizeof g_sharded_err, "%s: 1..%u keep thresholds", who, (unsigned)FASTF_SWEEP_MAX_RATES); return 1; }
    for (uint32_t i = 0; i < n_rates; i++)
        if (keep_thresholds[i] > 4294967296ull) { snprintf(g_sharded_err, sizeof g_sharded_err, "%s: keep_thresholds[%u] > 2^32", who, i); return 1; }
    const uint32_t K = n_rates;
    // sorted position p <-> caller index order[p]; ties keep caller order (a row's rate maps to the first of equal thresholds)
    std::vector<uint32_t> order(K), pos(K);
    std::vector<uint64_t> thr(K);
    for (uint32_t i = 0; i < K; i++) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return keep_thresholds[a] < keep_thresholds[b]; });
    for (uint32_t p = 0; p < K; p++) { thr[p] = keep_thresholds[order[p]]; pos[order[p]] = p; }
    fastf_bam2db_sweep_result sorted;
    if (run_shards(who, n_devices, devices, params, bgzf_bytes, n_bytes, K, thr.data(), &sorted)) return 1;
    *res = sorted;
    for (uint32_t i = 0; i < K; i++) res->rate[i] = sorted.rate[pos[i]];
    for (uint64_t r = 0; r < res->n_rows; r++) res->row_rate[r] = (uint8_t)order[res->row_rate[r]];
    return 0;
}
